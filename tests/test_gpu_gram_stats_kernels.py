"""Kernel-level references for the statistics stage: the tensor-core Gram (csrc/gram_tc.cu), the DMMA Gram
(csrc/suffstats.cu) and the glue from statistics to scores (centring, intercepts / evaluation vectors, quadratic forms in
csrc/solvers.cu and csrc/poisson_batch.cu).  Every entry point is called directly through its C ABI.

Tensor-core Gram: every output (analysis, plane counts, G) must have the BITS of the CPU model in
tests/gram_tc_reference.py, on an adversarial column catalogue (powers of two, first digits of 64, round-half-even ties,
-0.0, subnormals, columns needing more than 8 planes, maxima on both sides of the |E| < 900 switch, values near
DBL_MAX) used as columns of X and of Y.

fp64 kernels: compared with numpy longdouble (64-bit mantissa on x86-64).  A result passes when
|got - ref| <= C_ULP * n * u * mag, u = 2^-53, mag = the sum of |term| of the quantity, n = the longest chain of fp64
roundings one term passes through in the kernel (stated next to each test).  To first order such a chain of n
roundings contributes at most n u |term|; C_ULP = 4 leaves a factor of 4 over that for the second-order terms and
for the longdouble reference's own rounding (2^-64 per operation)."""
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
import gram_tc_reference as ref  # noqa: E402

LD = np.longdouble
U = 2.0 ** -53
C_ULP = 4
F64 = torch.float64
PAD_BITS = 0x7FF4DEADBEEF0001          # a signalling-NaN pattern in every padding element of an output


def _dev(a, dtype=F64):
    return torch.from_numpy(np.ascontiguousarray(a)).to(device="cuda", dtype=dtype)


def _st():
    return nat.stream_ptr()


def _p(a):
    return ctypes.c_void_p(a.ctypes.data)


def _ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _bits(a):
    a = a.detach().cpu().numpy() if torch.is_tensor(a) else np.asarray(a)
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def _same_bits(got, want, what):
    g, w = _bits(got), _bits(want)
    assert g.shape == w.shape, (what, g.shape, w.shape)
    bad = g != w
    if bad.any():
        i = np.unravel_index(np.argmax(bad), bad.shape)
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.size} differ; at {i}: got "
                             f"{g[i].view(np.float64)!r} ({int(g[i]):#x}), want {w[i].view(np.float64)!r} ({int(w[i]):#x})")


def _padded(shape):
    """Output buffer whose every element holds PAD_BITS."""
    return torch.full(shape, PAD_BITS, dtype=torch.int64, device="cuda").view(F64)


def _check(got, ref_val, bound, what):
    got = np.asarray(got, dtype=np.float64)
    err = np.abs(got.astype(LD) - ref_val)
    ok = err <= bound
    if not np.all(ok):
        i = np.unravel_index(np.argmin(np.where(ok, np.inf, -(err - bound).astype(np.float64))), err.shape)
        raise AssertionError(f"{what}: {np.count_nonzero(~ok)} of {ok.size} beyond the bound; at {i}: got {got[i]!r}, "
                             f"ref {float(ref_val[i])!r}, err {float(err[i]):.3e}, bound {float(bound[i]):.3e}")


def _bound(n, mag):
    return C_ULP * max(n, 1) * U * np.asarray(mag, dtype=LD)


# --------------------------------------------------------------------------- inputs
def _design(T, seed, n_x=None, photometry=8):
    """X = catalogue columns (+ synth_data photometry-like columns, + 0/1 event columns up to n_x), Y = two catalogue
    columns (ties, the column just above 2^900) and one photometry-like column."""
    rng = np.random.default_rng(seed)
    cols = ref.catalogue(T, rng)
    y_names = ["ties", "e901"]
    X = [v for k, v in cols.items() if k not in y_names]
    if T > 1:                                     # synth_base z-scores its columns
        X += list(synth_data.synth_base(T, photometry, seed).T)
    if n_x is not None:
        while len(X) < n_x:
            X.append((rng.random(T) < 0.1).astype(np.float64))
        X = X[:n_x]
    Y = [cols[k] for k in y_names] + [rng.standard_normal(T) * 3.0]
    return np.stack(X, axis=1), np.stack(Y, axis=1)


class Design:
    """X / Y on the device with row strides C + 1 / n_y + 2 (NaN in the gaps: a kernel that read them would show)."""

    def __init__(self, X, Y):
        self.X, self.Y = X, Y
        self.T, self.C = X.shape
        self.n_y = Y.shape[1]
        self.n_aug = self.C + self.n_y + 1
        bx = torch.full((self.T, self.C + 1), float("nan"), dtype=F64, device="cuda")
        bx[:, :self.C] = _dev(X)
        by = torch.full((self.T, self.n_y + 2), float("nan"), dtype=F64, device="cuda")
        by[:, :self.n_y] = _dev(Y)
        self.Xd, self.ldx, self.Yd, self.ldy = bx, self.C + 1, by, self.n_y + 2
        self.Z = ref.augment(X, Y)

    def args(self):
        return (_ptr(self.Xd), self.ldx, _ptr(self.Yd), self.ldy, self.n_y, self.T, self.C)


def _analyze(d, rs=None, max_planes=8):
    colE = torch.empty(d.n_aug, dtype=torch.int32, device="cuda")
    colS = torch.empty_like(colE)
    scratch = torch.empty(d.n_aug, dtype=torch.int64, device="cuda")
    flag = torch.empty(1, dtype=torch.int32, device="cuda")
    X, ldx, Y, ldy, n_y, T, C = d.args()
    if rs is None:
        nat.call("sglm_gram_tc_analyze_f64", X, ldx, Y, ldy, n_y, T, C, _ptr(colE), _ptr(colS), _ptr(scratch),
                 _ptr(flag), _st())
    else:
        nat.call("sglm_gram_tc_analyze_scaled_f64", X, ldx, Y, ldy, n_y, T, C, _ptr(rs), max_planes, _ptr(colE),
                 _ptr(colS), _ptr(scratch), _ptr(flag), _st())
    return colE, colS, int(flag.item())


def _colstats(d, rs=None):
    cm = torch.empty(d.n_aug, dtype=torch.int64, device="cuda")
    ls = torch.empty(d.n_aug, dtype=torch.int32, device="cuda")
    if rs is None:
        nat.call("sglm_gram_tc_colstats_f64", *d.args(), _ptr(cm), _ptr(ls), _st())
    else:
        nat.call("sglm_gram_tc_colstats_scaled_f64", *d.args(), _ptr(rs), _ptr(cm), _ptr(ls), _st())
    return cm, ls


def _exponents(cm, ls, max_planes=8):
    n = cm.numel()
    colE = torch.empty(n, dtype=torch.int32, device="cuda")
    colS = ls.clone()
    flag = torch.empty(1, dtype=torch.int32, device="cuda")
    nat.call("sglm_gram_tc_exponents", _ptr(cm), n, max_planes, _ptr(colE), _ptr(colS), _ptr(flag), _st())
    return colE, colS, int(flag.item())


def _rows(lists):
    """Concatenated row lists, each padded with -1 to a multiple of 128 (128 x -1 when there is none)."""
    parts = []
    for r in lists:
        parts += [np.asarray(r, dtype=np.int64), np.full((-len(r)) % 128, -1, dtype=np.int64)]
    a = np.concatenate(parts) if parts else np.zeros(0, dtype=np.int64)
    if a.size == 0:
        a = np.full(128, -1, dtype=np.int64)
    return _dev(a, torch.int64), np.ascontiguousarray([len(r) for r in lists], dtype=np.int64)


def _workspace(nbytes):
    raw = torch.empty(nbytes + 1024, dtype=torch.uint8, device="cuda")
    off = (-raw.data_ptr()) % 1024
    return raw, raw.data_ptr() + off


def _cells(sets, T):
    """Disjoint cells of the partition the (overlapping) sets induce, and member[o][c]."""
    sig = np.zeros(T, dtype=np.int64)
    for o, r in enumerate(sets):
        sig[np.asarray(r, dtype=np.int64)] |= 1 << o
    keys = [k for k in np.unique(sig) if k != 0]
    cells = [np.flatnonzero(sig == k) for k in keys]
    member = np.array([[(int(k) >> o) & 1 for k in keys] for o in range(len(sets))], dtype=np.int32)
    return cells, member


def _gram(d, colE, colS, sets, ldg, check=0, rs=None):
    colS_h = np.ascontiguousarray(colS.cpu().numpy(), dtype=np.int32)
    rows, sizes = _rows(sets)
    wb = nat.lib().sglm_gram_tc_workspace_bytes(d.n_aug, _p(colS_h), len(sets), _p(sizes))
    assert wb > 0
    raw, ws = _workspace(wb)
    G = _padded((len(sets), d.n_aug, ldg))
    X, ldx, Y, ldy, n_y, T, C = d.args()
    if rs is None:
        nat.call("sglm_gram_tc_f64", X, ldx, Y, ldy, n_y, T, C, _ptr(colE), _ptr(colS), _p(colS_h), len(sets), _p(sizes),
                 _ptr(rows), _ptr(G), ldg, ctypes.c_void_p(ws), wb, check, _st())
    else:
        nat.call("sglm_gram_tc_scaled_f64", X, ldx, Y, ldy, n_y, T, C, _ptr(rs), _ptr(colE), _ptr(colS), _p(colS_h),
                 len(sets), _p(sizes), _ptr(rows), _ptr(G), ldg, ctypes.c_void_p(ws), wb, _st())
    return G.cpu().numpy()


def _check_gram(G, want, n_aug, what):
    """G[:, :, :n_aug] has the model's bits, the padding columns up to ldg are untouched, G is exactly symmetric."""
    _same_bits(G[:, :, :n_aug], want, what)
    assert np.all(_bits(G[:, :, n_aug:]) == PAD_BITS), what + ": padding columns written"
    for g in G:
        assert np.array_equal(_bits(g[:, :n_aug]), _bits(g[:, :n_aug].T)), what + ": not symmetric"


def _plan_info(n_aug, colS_h, sizes):
    out = np.zeros(4, dtype=np.int64)
    assert nat.lib().sglm_gram_tc_plan_info(n_aug, _p(colS_h), len(sizes), _p(sizes), _p(out)) == 0
    return out


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


# --------------------------------------------------------------------------- 1. analysis
@pytest.mark.parametrize("T", [0, 1, 300, 5000])
def test_analysis_equals_model(T):
    d = Design(*_design(T, seed=T + 1))
    want = ref.analyze(d.Z)
    colE, colS, flag = _analyze(d)
    assert flag == want["flag"] == 0
    assert np.array_equal(colE.cpu().numpy(), want["colE"]) and np.array_equal(colS.cpu().numpy(), want["colS"])
    cm, ls = _colstats(d)
    assert np.array_equal(cm.cpu().numpy().view(np.uint64), want["colmax_bits"])
    assert np.array_equal(ls.cpu().numpy(), want["col_lsb"])
    e2, s2, f2 = _exponents(cm, ls)
    assert f2 == 0 and torch.equal(e2, colE) and torch.equal(s2, colS)
    rng = np.random.default_rng(T)
    rs = np.exp2(rng.integers(-20, 21, T)) * rng.uniform(1, 2, T)
    rs[::5] = 0.0
    rs_d = _dev(rs)
    for mp in range(1, 9):
        w = ref.analyze(d.Z, rs, mp)
        e, s, f = _analyze(d, rs_d, mp)
        assert f == w["flag"]                     # the column near DBL_MAX overflows once scaled by up to 2^21
        assert np.array_equal(e.cpu().numpy(), w["colE"]) and np.array_equal(s.cpu().numpy(), w["colS"]), mp
        cm, ls = _colstats(d, rs_d)
        assert np.array_equal(cm.cpu().numpy().view(np.uint64), w["colmax_bits"])
        assert np.array_equal(ls.cpu().numpy(), w["col_lsb"])
        e2, s2, _ = _exponents(cm, ls, mp)
        assert torch.equal(e2, e) and torch.equal(s2, s)


@pytest.mark.parametrize("where", ["X", "Y", "row_scale"])
@pytest.mark.parametrize("bad", [np.nan, np.inf, -np.inf])
def test_analysis_flags_non_finite(where, bad):
    """A NaN / inf in X, Y or row_scale: flag set, the column's max is the NaN pattern and it gets E = 0, S = 1.  The
    bad value sits in a column of ordinary values, whose lowest set bit decides col_lsb (the GPU's NaN payload can
    differ from numpy's)."""
    X, Y = _design(400, seed=3)
    rs = np.ones(400)
    if where == "X":
        X[17, -1] = bad
    elif where == "Y":
        Y[17, -1] = bad
    d = Design(X, Y)
    if where == "row_scale":
        rs[17] = bad
        e, s, f = _analyze(d, _dev(rs), 8)
        w = ref.analyze(d.Z, rs)
        cm, ls = _colstats(d, _dev(rs))
    else:
        e, s, f = _analyze(d)
        w = ref.analyze(d.Z)
        cm, ls = _colstats(d)
    assert f == w["flag"] == 1
    assert np.array_equal(e.cpu().numpy(), w["colE"]) and np.array_equal(s.cpu().numpy(), w["colS"])
    assert np.array_equal(cm.cpu().numpy().view(np.uint64), w["colmax_bits"])
    Zs = d.Z * rs[:, None]
    ordinary = np.any(np.isfinite(Zs) & (Zs != 0), axis=0)     # else col_lsb is the NaN's own lowest bit
    assert np.array_equal(ls.cpu().numpy()[ordinary], w["col_lsb"][ordinary])
    assert _exponents(cm, ls)[2] == 1


# --------------------------------------------------------------------------- 2. per-set Gram
@pytest.mark.parametrize("n_aug", [255, 256, 257, 513])
def test_gram_per_set_equals_model(n_aug):
    """Level 1 holds n_aug planes: 255 / 256 / 257 / 513 rows around the 256-row tiles.  Sets: full (T = 700, not a
    multiple of 128), empty, 1, 127, 128 and 129 rows; tcgen05 and the CUDA-core check GEMM."""
    T = 700
    X, Y = _design(T, seed=n_aug, n_x=n_aug - 4)
    d = Design(X, Y)
    assert d.n_aug == n_aug
    rng = np.random.default_rng(n_aug)
    sets = [np.arange(T), np.zeros(0, dtype=np.int64), np.array([T - 1])] + \
           [np.sort(rng.choice(T, k, replace=False)) for k in (127, 128, 129)]
    want, a = ref.gram(d.Z, sets)
    colE, colS, flag = _analyze(d)
    assert flag == 0 and np.array_equal(colS.cpu().numpy(), a["colS"])
    assert (a["colS"] == 8).any() and ref.plan(n_aug, a["colS"], [T])["level_cnt"][1] == n_aug
    ldg = n_aug + 3
    for check in (0, 1):
        G = _gram(d, colE, colS, sets, ldg, check=check)
        _check_gram(G, want, n_aug, f"n_aug={n_aug} check_gemm={check}")
    info = _plan_info(n_aug, a["colS"].astype(np.int32), np.array([len(s) for s in sets], dtype=np.int64))
    p = ref.plan(n_aug, a["colS"], [len(s) for s in sets], sms=_sms())
    assert list(info) == [p["S"], p["n_pos"], len(p["tiles"]), p["n_parts"]]


def test_gram_several_k_parts_equals_model():
    """Sets large enough for the plan to cut K into several parts (asserted from plan_info): part boundaries fall
    inside sets, each part drains its own int32 accumulators."""
    T = 60000
    rng = np.random.default_rng(11)
    X = rng.standard_normal((T, 60))
    X[:, :4] = ref.augment(*_design(T, seed=12))[:, :4]
    Y = rng.standard_normal((T, 1))
    d = Design(X, Y)
    sets = [np.arange(T), np.sort(rng.choice(T, 20000, replace=False)), np.arange(5, T, 7)]
    want, a = ref.gram(d.Z, sets)
    sizes = np.array([len(s) for s in sets], dtype=np.int64)
    info = _plan_info(d.n_aug, a["colS"].astype(np.int32), sizes)
    assert info[3] > 1, info
    assert info[3] == ref.plan(d.n_aug, a["colS"], sizes, sms=_sms())["n_parts"]
    colE, colS, _ = _analyze(d)
    _check_gram(_gram(d, colE, colS, sets, d.n_aug + 1), want, d.n_aug, "K parts")


# --------------------------------------------------------------------------- 3. cells
def test_cells_and_partial_cells_equal_model():
    T = 3000
    d = Design(*_design(T, seed=21))
    rng = np.random.default_rng(21)
    sets = [np.arange(T)] + [np.sort(rng.choice(T, n, replace=False)) for n in (600, 900, 1500, 2400)]
    want, a = ref.gram(d.Z, sets)
    colE, colS, _ = _analyze(d)
    colS_h = np.ascontiguousarray(colS.cpu().numpy(), dtype=np.int32)
    cells, member = _cells(sets, T)
    n_out = len(sets)
    ldg = d.n_aug + 2
    member = np.ascontiguousarray(member)
    for check in (0, 1):
        rows, sizes = _rows(cells)
        wb = nat.lib().sglm_gram_tc_cells_workspace_bytes(d.n_aug, _p(colS_h), len(cells), _p(sizes), n_out)
        raw, ws = _workspace(wb)
        G = _padded((n_out, d.n_aug, ldg))
        nat.call("sglm_gram_tc_cells_f64", *d.args(), _ptr(colE), _ptr(colS), _p(colS_h), len(cells), _p(sizes),
                 _ptr(rows), n_out, _p(member), _ptr(G), ldg, ctypes.c_void_p(ws), wb, check, _st())
        _check_gram(G.cpu().numpy(), want, d.n_aug, f"cells check_gemm={check}")
    # row-sharded form: three random row partitions, int64 plane Grams summed on the host, then combine
    part_of = rng.integers(0, 3, T)
    total = None
    for p in range(3):
        mine = [c[part_of[c] == p] for c in cells]
        rows, sizes = _rows(mine)
        wb = nat.lib().sglm_gram_tc_cells_workspace_bytes(d.n_aug, _p(colS_h), len(mine), _p(sizes), n_out)
        raw, ws = _workspace(wb)
        nat.call("sglm_gram_tc_cells_partial_f64", *d.args(), _ptr(colE), _ptr(colS), _p(colS_h), len(mine), _p(sizes),
                 _ptr(rows), n_out, _p(member), ctypes.c_void_p(ws), wb, _st())
        off, size = ctypes.c_uint64(0), ctypes.c_uint64(0)
        assert nat.lib().sglm_gram_tc_cells_sgout(d.n_aug, _p(colS_h), len(mine), _p(sizes), n_out, ctypes.byref(off),
                                                  ctypes.byref(size)) == 0
        sg = raw[ws - raw.data_ptr() + off.value: ws - raw.data_ptr() + off.value + size.value].view(torch.int64).clone()
        total = sg if total is None else total + sg
    G = _combine(d, colE, colS, colS_h, cells, n_out, total, ldg)
    _check_gram(G, want, d.n_aug, "partial cells + combine")


def _combine(d, colE, colS, colS_h, cells, n_out, sg_sum, ldg, C=None):
    rows, sizes = _rows(cells)
    wb = nat.lib().sglm_gram_tc_cells_workspace_bytes(d.n_aug, _p(colS_h), len(cells), _p(sizes), n_out)
    raw, ws = _workspace(wb)
    off, size = ctypes.c_uint64(0), ctypes.c_uint64(0)
    assert nat.lib().sglm_gram_tc_cells_sgout(d.n_aug, _p(colS_h), len(cells), _p(sizes), n_out, ctypes.byref(off),
                                              ctypes.byref(size)) == 0
    assert size.value == sg_sum.numel() * 8
    o = ws - raw.data_ptr() + off.value
    raw[o:o + size.value].view(torch.int64).copy_(sg_sum)
    G = _padded((n_out, d.n_aug, ldg))
    nat.call("sglm_gram_tc_cells_combine_f64", d.C if C is None else C, d.n_y, _ptr(colE), _ptr(colS), _p(colS_h),
             len(cells), _p(sizes), n_out, _ptr(G), ldg, ctypes.c_void_p(ws), wb, _st())
    return G.cpu().numpy()


# --------------------------------------------------------------------------- 4. int32 drain boundary
V2 = 63.5 / 64                                       # digits [64, -64]
V3 = (63.5 + 0.5 / 128) / 64                         # digits [64, -64, 64]


def _all_64_design(T):
    """Columns whose digits are all +-64 (|d d'| = 2^12 on every row, the largest per-row product)."""
    t = np.arange(T)
    X = np.stack([np.full(T, V2), np.full(T, V3), np.where(t % 2 == 0, V3, -V3)], axis=1)
    return Design(X, np.full((T, 1), -V2))


def test_drain_boundary_equals_model():
    """One set of 2048 * 128 + 1 rows (a 2048-block K segment and a 1-block one) and one of 2 * 2048 * 128 rows, whose
    set Gram of 2^31 only the int64 drain holds.  The plan cuts K into parts here, so a segment boundary falls inside
    a part; test_full_segment_in_one_k_part fills one int32 accumulator to the limit."""
    T = 2 * 2048 * 128
    d = _all_64_design(T)
    for c in range(4):
        a = ref.analyze(d.Z[:5, c:c + 1])
        p = ref.digits(d.Z[:5, c:c + 1], None, a["colE"], a["colS"])[0]
        assert np.all(np.abs(p) == 64)
    sets = [np.arange(2048 * 128 + 1), np.arange(T)]
    want, a = ref.gram(d.Z, sets)
    assert want[1, 0, 0] == T * V2 * V2
    colE, colS, _ = _analyze(d)
    _check_gram(_gram(d, colE, colS, sets, d.n_aug), want, d.n_aug, "drain boundary")


def test_full_segment_in_one_k_part():
    """The int32 accumulators of the tcgen05 GEMM are drained at every K segment boundary and every K part boundary.
    One set of 16 * 2 * 2048 * 128 rows: the plan (asserted from plan_info) cuts K into 16 parts of 4096 blocks, so every
    part holds two whole segments of TC_MAX_KB_PER_SEG = 2048 blocks, and the level-1 plane Gram of the constant column
    reaches 2048 * 128 * 2^12 = 2^30 in one accumulator.  A segment cut at more than 2048 blocks would overflow int32
    there.  The columns are constant or alternate in sign, so the exact Gram is (T / 2) times the Gram of two rows."""
    kb = 16 * 2 * ref.TC_MAX_KB_PER_SEG
    T = kb * ref.TC_BK
    d = _all_64_design(T)
    colE, colS, flag = _analyze(d)
    assert flag == 0
    colS_h = np.ascontiguousarray(colS.cpu().numpy(), dtype=np.int32)
    sizes = np.array([T], dtype=np.int64)
    info = _plan_info(d.n_aug, colS_h, sizes)
    p = ref.plan(d.n_aug, colS_h, [T], sms=_sms())
    assert list(info) == [p["S"], p["n_pos"], len(p["tiles"]), p["n_parts"]]
    assert info[3] == 16, info
    for part in range(p["n_parts"]):
        lo, hi = kb * part // p["n_parts"], kb * (part + 1) // p["n_parts"]
        assert any(s[1] == ref.TC_MAX_KB_PER_SEG and lo <= s[0] and s[0] + s[1] <= hi for s in p["segs"]), part
    two = d.Z[:2]
    want = (two.T @ two) * (T // 2)                 # exact: few-bit dyadic products times a power of two
    G = _gram(d, colE, colS, [np.arange(T)], d.n_aug)
    _check_gram(G, want[None], d.n_aug, "full segment in one K part")


# --------------------------------------------------------------------------- 5. weighted Gram
@pytest.mark.parametrize("max_planes", sorted({1, 2, eng.POISSON_TC_PLANES, 8}))
def test_weighted_gram_equals_model_and_bound(max_planes):
    T = 1500
    d = Design(*_design(T, seed=31 + max_planes))
    rng = np.random.default_rng(max_planes)
    rs = np.exp2(rng.integers(-20, 21, T)) * rng.uniform(1, 2, T)
    rs[rng.choice(T, 100, replace=False)] = 0.0
    # the column near DBL_MAX overflows once scaled; drop it from the weighted design
    keep = [c for c in range(d.C) if np.all(np.isfinite(d.X[:, c] * rs))]
    d = Design(d.X[:, keep], d.Y)
    rs_d = _dev(rs)
    sets = [np.arange(T), np.sort(rng.choice(T, 700, replace=False))]
    want, a = ref.gram(d.Z, sets, rs=rs, max_planes=max_planes)
    colE, colS, flag = _analyze(d, rs_d, max_planes)
    assert flag == 0 and np.array_equal(colS.cpu().numpy(), a["colS"])
    G = _gram(d, colE, colS, sets, d.n_aug + 1, rs=rs_d)
    _check_gram(G, want, d.n_aug, f"scaled max_planes={max_planes}")
    # row-sharded weighted form: colstats_scaled + exponents, three partitions of partials, combine
    cm, ls = _colstats(d, rs_d)
    e2, s2, _ = _exponents(cm, ls, max_planes)
    assert torch.equal(e2, colE) and torch.equal(s2, colS)
    colS_h = np.ascontiguousarray(colS.cpu().numpy(), dtype=np.int32)
    member = np.eye(len(sets), dtype=np.int32)
    part_of = rng.integers(0, 3, T)
    total = None
    for p in range(3):
        mine = [s[part_of[s] == p] for s in sets]
        rows, sizes = _rows(mine)
        wb = nat.lib().sglm_gram_tc_cells_workspace_bytes(d.n_aug, _p(colS_h), len(mine), _p(sizes), len(sets))
        raw, ws = _workspace(wb)
        nat.call("sglm_gram_tc_scaled_partial_f64", *d.args(), _ptr(rs_d), _ptr(colE), _ptr(colS), _p(colS_h), len(mine),
                 _p(sizes), _ptr(rows), len(sets), _p(member), ctypes.c_void_p(ws), wb, _st())
        off, size = ctypes.c_uint64(0), ctypes.c_uint64(0)
        nat.lib().sglm_gram_tc_cells_sgout(d.n_aug, _p(colS_h), len(mine), _p(sizes), len(sets), ctypes.byref(off),
                                           ctypes.byref(size))
        sg = raw[ws - raw.data_ptr() + off.value: ws - raw.data_ptr() + off.value + size.value].view(torch.int64).clone()
        total = sg if total is None else total + sg
    _check_gram(_combine(d, colE, colS, colS_h, sets, len(sets), total, d.n_aug + 1), want, d.n_aug,
                f"scaled partial + combine, max_planes={max_planes}")
    # documented accuracy, independent of the model: against the Gram of the fp64 products zr = z * rs,
    # |dG_ij| <= sum_t (|zr_ti| delta_j + |zr_tj| delta_i + delta_i delta_j) + dropped k + l > 9 pairs + 9 u sum|zr_i zr_j|,
    # delta_c = 2^(E_c - 7 S_c) when the column needs more than S_c planes (else 0); the longdouble reference adds
    # T 2^-63 sum|zr_i zr_j|
    Zr = d.Z * rs[:, None]
    E, S = a["colE"].astype(np.int64), a["colS"].astype(np.int64)
    need = ref.exponents(a["colmax_bits"], a["col_lsb"], 99)[1]
    delta = np.where(need > S, np.exp2((E - 7 * S).astype(LD)), LD(0))
    planes = ref.digits(d.Z, rs, a["colE"], a["colS"])
    for s, rows in enumerate(sets):
        Zl = np.abs(Zr[rows]).astype(LD)
        exact = Zr[rows].astype(LD).T @ Zr[rows].astype(LD)
        absg = Zl.T @ Zl
        colsum = Zl.sum(axis=0)
        dropped = np.zeros((d.n_aug, d.n_aug), dtype=LD)
        lev = [np.stack([np.abs(p[k, rows]).astype(np.float64) if p.shape[0] > k else np.zeros(len(rows))
                         for p in planes], axis=1) * 2.0 ** (-6 - 7 * k) for k in range(8)]
        for k in range(8):
            for l in range(8):
                if k + l + 2 > 9:
                    dropped += (lev[k].T @ lev[l]).astype(LD)
        dropped *= np.exp2((E[:, None] + E[None, :]).astype(LD))
        bound = (colsum[:, None] * delta[None, :] + colsum[None, :] * delta[:, None] + len(rows) * np.outer(delta, delta)
                 + dropped + (9 * U + len(rows) * 2.0 ** -63) * absg + LD(2.0 ** -1074))   # + subnormal results
        bound = np.where(absg > ref.DBL_MAX / 2, LD(np.inf), bound)  # entries that overflow fp64 (inf in G) are not bounded
        _check(G[s, :, :d.n_aug], exact, bound, f"weighted accuracy, max_planes={max_planes}, set {s}")


# --------------------------------------------------------------------------- 6. lag design
@pytest.mark.parametrize("n_out", [0, 3])
def test_lag_gram_equals_model(n_out):
    """Lag columns read base[t + off_c, src_c]: offsets 0 .. n_u - T, i.e. shifts of both signs around the middle;
    base signal 0 has its extreme value in the window's first row, base signal 1 in its last row."""
    rng = np.random.default_rng(41 + n_out)
    T, h, P = 900, 6, 5
    n_u = T + 2 * h
    base = synth_data.synth_base(n_u, P, 41)
    base[:, 2] = ref.catalogue(n_u, rng)["ties"]
    base[:, 3] = ref.catalogue(n_u, rng)["one_plus_tiny"]
    base[0, 0] = 40.0 * np.abs(base[:, 0]).max()
    base[-1, 1] = -40.0 * np.abs(base[:, 1]).max()
    src = np.repeat(np.arange(P), 2 * h + 1).astype(np.int32)
    off = np.tile(np.arange(2 * h + 1), P).astype(np.int32)          # off = h -> shift 0
    C = len(src)
    Y = np.stack([rng.standard_normal(T), ref.catalogue(T, rng)["first_digit_64"]], axis=1)
    n_y = Y.shape[1]
    n_aug = C + n_y + 1
    sets = [np.arange(T), np.sort(rng.choice(T, 300, replace=False)), np.arange(0, T, 2)]
    want, colE_m, colS_m = ref.lag_gram(base, src, off, Y, sets)
    # analysis of [base | 1] over the window and of [Y | 1] (colstats + exponents, as _engine._lag_analysis)
    bw = _dev(base)
    Yd = _dev(Y)
    cm_b = torch.empty(P + 1, dtype=torch.int64, device="cuda")
    ls_b = torch.empty(P + 1, dtype=torch.int32, device="cuda")
    nat.call("sglm_gram_tc_colstats_f64", _ptr(bw), P, None, 0, 0, n_u, P, _ptr(cm_b), _ptr(ls_b), _st())
    bE, bS, f1 = _exponents(cm_b, ls_b)
    cm_y = torch.empty(n_y + 1, dtype=torch.int64, device="cuda")
    ls_y = torch.empty(n_y + 1, dtype=torch.int32, device="cuda")
    nat.call("sglm_gram_tc_colstats_f64", None, 0, _ptr(Yd), n_y, n_y, T, 0, _ptr(cm_y), _ptr(ls_y), _st())
    yE, yS, f2 = _exponents(cm_y, ls_y)
    assert f1 == f2 == 0
    src_t = _dev(src, torch.int64)
    colE = torch.cat([bE.index_select(0, src_t), yE]).contiguous()
    colS = torch.cat([bS.index_select(0, src_t), yS]).contiguous()
    assert np.array_equal(colE.cpu().numpy(), colE_m) and np.array_equal(colS.cpu().numpy(), colS_m)
    colS_h = np.ascontiguousarray(colS.cpu().numpy(), dtype=np.int32)
    bS_h = np.ascontiguousarray(bS.cpu().numpy(), dtype=np.int32)
    if n_out == 0:
        lists, member = sets, None
    else:
        lists, member = _cells(sets, T)
    rows, sizes = _rows(lists)
    desc = nat.LagDesignStruct(bw.data_ptr(), P, n_u, P, src.ctypes.data, off.ctypes.data, bE.data_ptr(), bS.data_ptr(),
                               bS_h.ctypes.data)
    wb = nat.lib().sglm_gram_tc_lag_workspace_bytes(n_aug, _p(colS_h), len(lists), _p(sizes), n_out, P, _p(bS_h), n_u)
    assert wb > 0
    raw, ws = _workspace(wb)
    ldg = n_aug + 1
    G = _padded((len(sets), n_aug, ldg))
    nat.call("sglm_gram_tc_lag_cells_f64", ctypes.byref(desc), _ptr(Yd), n_y, n_y, T, C, _ptr(colE), _ptr(colS),
             _p(colS_h), len(lists), _p(sizes), _ptr(rows), n_out, None if member is None else _p(member), _ptr(G), ldg,
             ctypes.c_void_p(ws), wb, 0, _st())
    _check_gram(G.cpu().numpy(), want, n_aug, f"lag n_out={n_out}")
    if n_out:
        raw2, ws2 = _workspace(wb)
        nat.call("sglm_gram_tc_lag_cells_f64", ctypes.byref(desc), _ptr(Yd), n_y, n_y, T, C, _ptr(colE), _ptr(colS),
                 _p(colS_h), len(lists), _p(sizes), _ptr(rows), n_out, _p(member), None, ldg, ctypes.c_void_p(ws2), wb, 1,
                 _st())
        G2 = _padded((len(sets), n_aug, ldg))
        nat.call("sglm_gram_tc_cells_combine_f64", C, n_y, _ptr(colE), _ptr(colS), _p(colS_h), len(lists), _p(sizes),
                 n_out, _ptr(G2), ldg, ctypes.c_void_p(ws2), wb, _st())
        _check_gram(G2.cpu().numpy(), want, n_aug, "lag partial + combine")


# --------------------------------------------------------------------------- 7. DMMA statistics
def _suffstats(d, W, ks, ldg):
    n_sets = 1 if W is None else W.shape[0]
    ks = np.ascontiguousarray(ks, dtype=np.int32)
    wb = nat.lib().sglm_suffstats_workspace_bytes(d.T, d.C, d.n_y, n_sets, _p(ks))
    assert wb > 0
    ws = torch.empty((wb + 255) // 256 * 32, dtype=F64, device="cuda")
    G = _padded((n_sets, d.n_aug, ldg))
    nat.call("sglm_suffstats_f64", *d.args()[:5], d.T, d.C, _ptr(W), 0 if W is None else W.stride(0), n_sets, _p(ks),
             _ptr(G), ldg, _ptr(ws), ws.numel() * 8, _st())
    return G.cpu().numpy()


@pytest.mark.parametrize("ks", [1, 3, 16])
def test_suffstats_dmma_against_longdouble(ks):
    """Bound: a term w z_i z_j passes through the product w z_i (1 rounding), at most T accumulations inside the
    K chunk and ks chunk sums: n = T + ks + 1."""
    T = 2000
    X, Y = _design(T, seed=51)
    keep = [c for c in range(X.shape[1]) if np.abs(X[:, c]).max() < 1e100 and np.abs(X[:, c]).max() > 1e-100]
    X = X[:, keep]
    Y = Y[:, [0, 2]]
    d = Design(X, Y)
    rng = np.random.default_rng(ks)
    W = np.stack([(rng.random(T) < 0.4).astype(np.float64), rng.integers(0, 4, T).astype(np.float64), np.zeros(T),
                  rng.uniform(0, 3, T)])
    Wd = torch.zeros((4, T + 5), dtype=F64, device="cuda")
    Wd[:, :T] = _dev(W)
    ldg = d.n_aug + 1
    G = _suffstats(d, Wd, [ks] * 4, ldg)
    G1 = _suffstats(d, None, [ks], ldg)
    for s, w in enumerate(list(W) + [None]):
        g = G1[0] if w is None else G[s]
        refv, mag = ref.suffstats_dmma(d.Z, w)
        _check(g[:, :d.n_aug], refv, _bound(T + ks + 1, mag), f"suffstats set {s} ks={ks}")
        assert np.all(_bits(g[:, d.n_aug:]) == PAD_BITS)
        assert np.array_equal(_bits(g[:, :d.n_aug]), _bits(g[:, :d.n_aug].T))
    assert not G[2, :, :d.n_aug].any()                                    # all-zero weights
    _same_bits(_suffstats(d, Wd, [ks] * 4, ldg), G, f"suffstats repeat ks={ks}")


def test_suffstats_exact_data_equals_tc_gram():
    """Small integers with T max^2 < 2^53: every partial sum of the DMMA Gram is exact, and so is the tensor-core
    Gram (S1 + S2 <= 9), so both have the bits of Z'Z."""
    T = 3000
    rng = np.random.default_rng(61)
    X = np.concatenate([rng.integers(-100, 101, (T, 6)), (rng.random((T, 4)) < 0.3)], axis=1).astype(np.float64)
    Y = rng.integers(0, 50, (T, 1)).astype(np.float64)
    d = Design(X, Y)
    want, a = ref.gram(d.Z, [np.arange(T)])
    assert np.array_equal(want[0], d.Z.T @ d.Z)
    for ks in (1, 5):
        G = _suffstats(d, None, [ks], d.n_aug)
        _same_bits(G, want, f"DMMA Gram on exact data, ks={ks}")


def test_index_counts_exact():
    T = 5000
    rng = np.random.default_rng(71)
    idx = np.concatenate([rng.integers(0, T, 20000), rng.integers(-T, 0, 3000), np.full(50, 7), np.full(30, -1)])
    counts = torch.zeros(T, dtype=F64, device="cuda")
    it = _dev(idx, torch.int64)
    nat.call("sglm_index_counts_f64", _ptr(it), it.numel(), _ptr(counts), T, _st())
    want = np.bincount(np.where(idx < 0, idx + T, idx), minlength=T).astype(np.float64)
    _same_bits(counts, want, "index counts")


# --------------------------------------------------------------------------- 8. centring
def _center(Ap, Am, C, n_y, y_col, fit, ldq):
    ldg = Ap.shape[1]
    Apd = _dev(Ap)
    Amd = None if Am is None else _dev(Am)
    Qc = _padded((C, ldq))
    qc, xbar, diag = _padded((C,)), _padded((C,)), _padded((C,))
    scal = _padded((4,))
    nat.call("sglm_center_stats_f64", _ptr(Apd), _ptr(Amd), ldg, C, n_y, y_col, fit, _ptr(Qc), ldq, _ptr(qc), _ptr(xbar),
             _ptr(diag), _ptr(scal), _st())
    return [t.cpu().numpy() for t in (Qc, qc, xbar, diag, scal)]


def _stats(T, C, n_y, seed, mean=0.0):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((T, C)) + mean
    Y = rng.standard_normal((T, n_y)) + 2.0
    Z = ref.augment(X, Y)
    full = (Z.T @ Z)
    test = np.sort(rng.choice(T, T // 5, replace=False))
    return Z, full, Z[test].T @ Z[test]


N_CENTER = 8          # rounding chain of the centred entries (test_center_stats_against_longdouble)


@pytest.mark.parametrize("minus", [False, True])
@pytest.mark.parametrize("fit", [1, 0])
def test_center_stats_against_longdouble(minus, fit):
    """mag = |A+_ij| + |A-_ij| + n |xbar_i xbar_j|.  Chains (N_CENTER = 8 for Qc / qc / yyc): the n xbar_i xbar_j term
    passes through the subtractions A+ - A- giving n, A_i1 and A_j1, the two divisions, the two products and the final
    difference (8 roundings); the A_ij term through its subtraction and the final difference (2).  xbar / ybar: the two
    subtractions and the division (3); sum y: one subtraction (1)."""
    C, n_y, y_col = 37, 3, 1
    Z, Ap, Am = _stats(800, C, n_y, seed=81)
    Am = Am if minus else None
    ldq = C + 5
    Qc, qc, xbar, diag, scal = _center(np.pad(Ap, ((0, 0), (0, 2))), None if Am is None else np.pad(Am, ((0, 0), (0, 2))),
                                       C, n_y, y_col, fit, ldq)
    r = ref.center(Ap, Am, C, n_y, y_col, bool(fit))
    _check(Qc[:, :C], r["Qc"][0], _bound(N_CENTER, r["Qc"][1]), "Qc")
    _check(qc, r["qc"][0], _bound(N_CENTER, r["qc"][1]), "qc")
    _check(xbar, r["xbar"][0], _bound(3, r["xbar"][1]), "xbar")
    _check(scal[[0]], np.array([r["yyc"][0]]), _bound(N_CENTER, [r["yyc"][1]]), "yyc")
    _check(scal[[2]], np.array([r["ybar"][0]]), _bound(3, [r["ybar"][1]]), "ybar")
    _check(scal[[3]], np.array([r["sy"][0]]), _bound(1, [r["sy"][1]]), "sum y")
    one = C + n_y
    n = Ap[one, one] - (Am[one, one] if Am is not None else 0.0)
    _same_bits(scal[[1]], np.array([n]), "scal[1] == n")
    _same_bits(diag, np.diag(Qc[:, :C]).copy(), "diag")
    assert not Qc[:, C:].any() and not np.signbit(Qc[:, C:]).any(), "columns C..ldq-1 of Qc"
    if not fit:
        want = Ap[:C, :C] - (Am[:C, :C] if Am is not None else 0.0)
        _same_bits(Qc[:, :C], want, "Qc without centring")


def test_center_stats_cancellation_bound():
    """A column of mean 1e3 and standard deviation 1: A_ii - n xbar_i^2 cancels ~6 decimal digits.  Pinned as a
    documented bound, not an accuracy claim: against the exactly centred Gram, relative error
    <= 2 C_ULP N_CENTER u (1 + mean^2 / var) (the bound above, whose mag is about 2 n (mean^2 + var), divided by
    n var; it also covers the rounding of A itself), here ~7e-9."""
    C, n_y = 4, 1
    T = 1000
    mean = 1e3
    rng = np.random.default_rng(91)
    X = rng.standard_normal((T, C))
    X = (X - X.mean(axis=0)) / X.std(axis=0) + mean
    Y = rng.standard_normal((T, 1))
    Z = ref.augment(X, Y)
    Zl = Z.astype(LD)
    Ap = (Zl.T @ Zl).astype(np.float64)
    Qc, *_ = _center(Ap, None, C, n_y, 0, 1, C)
    Xc = X.astype(LD) - X.astype(LD).mean(axis=0)
    exact = Xc.T @ Xc
    var = np.diag(exact) / T
    rel = np.abs(Qc.astype(LD) - exact) / np.sqrt(np.outer(np.diag(exact), np.diag(exact)))
    bound = 2 * C_ULP * N_CENTER * U * (1 + mean ** 2 / np.sqrt(np.outer(var, var)))
    assert np.all(rel <= bound), (float(rel.max()), float(bound.max()))


# --------------------------------------------------------------------------- 9. intercepts and evaluation vectors
@pytest.mark.parametrize("with_xbar", [True, False])
def test_finalize_models(with_xbar):
    """Bound for b: n = C + 1 (the strided per-thread sums, the warp tree, the four warp partials and ybar - s)."""
    C, n_y, n_models = 300, 3, 9
    ldw, ldv = C + 3, C + n_y + 1 + 4
    rng = np.random.default_rng(101)
    W = rng.standard_normal((n_models, ldw)) * np.exp2(rng.integers(-10, 11, (n_models, ldw)))
    W[:, C:] = np.nan
    n_prob = 3
    xb = rng.standard_normal((n_prob, C)) * 5.0
    yb = rng.standard_normal(n_prob)
    prob = rng.integers(0, n_prob, n_models)
    y_col = rng.integers(0, n_y, n_models).astype(np.int32)
    Wd, xbd = _dev(W), _dev(xb)
    xptr = _dev(np.array([xbd[p].data_ptr() for p in prob], dtype=np.int64), torch.int64)
    ybd = _dev(yb[prob])
    ycd = _dev(y_col, torch.int32)
    b = _padded((n_models,))
    V = _padded((n_models, ldv))
    nat.call("sglm_finalize_models_f64", _ptr(Wd), ldw, C, n_y, _ptr(ycd), _ptr(xptr) if with_xbar else None,
             _ptr(ybd) if with_xbar else None, n_models, _ptr(b), _ptr(V), ldv, _st())
    b, V = b.cpu().numpy(), V.cpu().numpy()
    if with_xbar:
        rb, mag = ref.finalize(W[:, :C], xb[prob], yb[prob])
        _check(b, rb, _bound(C + 1, mag), "intercept")
    else:
        assert np.all(_bits(b) == 0)
    _same_bits(V[:, :C], -W[:, :C], "V[:C] = -w")
    ey = np.zeros((n_models, n_y))
    ey[np.arange(n_models), y_col] = 1.0
    _same_bits(V[:, C:C + n_y], ey, "e_y")
    _same_bits(V[:, C + n_y], -b, "V[C + n_y] = -b")
    assert np.all(_bits(V[:, C + n_y + 1:]) == 0)


# --------------------------------------------------------------------------- 10. quadratic forms
def _sym(n, rng):
    A = rng.standard_normal((n, n))
    return A + A.T


@pytest.mark.parametrize("n,n_models", [(100, 20), (100, 5), (3300, 9)])
def test_quadform_against_longdouble(n, n_models):
    """mb = 8 (n <= 3200 and at least 8 models) and mb = 4 (fewer models, or n > 3200).  Bound n_chain = n + 32: a
    term passes through at most n / 32 lane sums, the products by A and v_i, n / 8 row sums per warp, 5 shuffle
    levels, 8 warp partials and up to 16 split partials."""
    rng = np.random.default_rng(n + n_models)
    lda, ldv = n + 1, n + 2
    A = np.full((n, lda), np.nan)
    A[:, :n] = _sym(n, rng)
    V = np.full((n_models, ldv), np.nan)
    V[:, :n] = rng.standard_normal((n_models, n))
    Ad, Vd = _dev(A), _dev(V)
    out = _padded((n_models,))
    nat.call("sglm_quadform_f64", _ptr(Ad), lda, n, _ptr(Vd), ldv, n_models, _ptr(out), _st())
    r, mag = ref.quadform(A[:, :n], V[:, :n])
    _check(out.cpu().numpy(), r, _bound(n + 32, mag), "quadform")
    again = _padded((n_models,))
    nat.call("sglm_quadform_f64", _ptr(Ad), lda, n, _ptr(Vd), ldv, n_models, _ptr(again), _st())
    _same_bits(again, out, "quadform repeat")
    for splits in (1, 3, 16):
        part = _padded((splits, n_models))
        nat.call("sglm_quadform_split_f64", _ptr(Ad), lda, n, _ptr(Vd), ldv, n_models, splits, _ptr(part), _st())
        p = part.cpu().numpy()
        s = p[0].copy()
        for k in range(1, splits):
            s = s + p[k]
        _check(s, r, _bound(n + 32, mag), f"quadform split {splits}")


@pytest.mark.parametrize("n_models", [1, 63, 64, 65, 200])
def test_quadform_gemm_against_longdouble(n_models):
    """Bound n_chain = 2 n + 16: the GEMM's k sum (n), the column dot's 16 row chunks (n / 16 fma each) and the 16
    chunk partials.  A model's result does not depend on the other models of the batch."""
    n = 333
    rng = np.random.default_rng(n_models)
    A = _sym(n, rng)
    ldb = (n_models + 63) // 64 * 64
    V = rng.standard_normal((n_models, n))
    Vt = np.zeros((n, ldb))
    Vt[:, :n_models] = V.T
    Ad, Vtd = _dev(A), _dev(Vt)
    Yw = torch.empty((n, ldb), dtype=F64, device="cuda")
    part = torch.empty((16, n_models), dtype=F64, device="cuda")
    out = _padded((n_models,))
    nat.call("sglm_quadform_gemm_f64", _ptr(Ad), n, n, _ptr(Vtd), ldb, n_models, _ptr(Yw), _ptr(part), _ptr(out), _st())
    r, mag = ref.quadform(A, V)
    _check(out.cpu().numpy(), r, _bound(2 * n + 16, mag), "quadform gemm")
    again = _padded((n_models,))
    nat.call("sglm_quadform_gemm_f64", _ptr(Ad), n, n, _ptr(Vtd), ldb, n_models, _ptr(Yw), _ptr(part), _ptr(again), _st())
    _same_bits(again, out, "quadform gemm repeat")
    for m in sorted({0, n_models // 2, n_models - 1}):
        one = np.zeros((n, 64))
        one[:, 0] = V[m]
        o1 = _padded((1,))
        nat.call("sglm_quadform_gemm_f64", _ptr(Ad), n, n, _ptr(_dev(one)), 64, 1, _ptr(Yw), _ptr(part), _ptr(o1), _st())
        _same_bits(o1, out[m:m + 1], f"quadform gemm model {m} alone")


def test_quadform_too_large_is_unsupported():
    n = 227 * 1024 // 32 + 1
    A = torch.zeros(8, dtype=F64, device="cuda")
    out = torch.zeros(8, dtype=F64, device="cuda")
    lib = nat.lib()
    assert lib.sglm_quadform_f64(_ptr(A), n, n, _ptr(A), n, 3, _ptr(out), _st()) == -6
    assert lib.sglm_quadform_split_f64(_ptr(A), n, n, _ptr(A), n, 3, 2, _ptr(out), _st()) == -6
