"""
Device-side orchestration of the sGLM hot path on one B200.

Everything numeric happens in libsglm_b200.so (hand-written sm_100a kernels, see
csrc/ and include/sglm_b200.h); this module only owns device buffers (torch tensors),
the launch plan and the small host<->device transfers.  There is no CPU fallback.

Launch plan for a CV grid (reference: backend/sglm_cv.py:42-428 — one sklearn fit per
(param set, fold) from 4 Python threads, X[idx,:] copied per fold):

  1. one pass over X per row set builds the augmented statistics G[s] = Z'diag(w_s)Z,
     Z = [X | Y | 1]  (full data + each test fold; train = full - test, no fold copies);
  2. per (fold, y column, fit_intercept) a centred problem (Qc, qc, yyc) is derived;
  3. ALL ElasticNet/Lasso models of the grid run in ONE batched coordinate-descent launch
     (one CTA per model), Ridge/OLS models in one Cholesky launch per problem;
  4. intercepts, train/test RSS and TSS come from the statistics (quadratic forms), so
     no model ever re-reads X.
"""
import ctypes

import numpy as np

import _sglm_native as nat
from _sglm_native import call, ptr, stream_ptr

_SM_TARGET_ITEMS = 148 * 8


# --------------------------------------------------------------------------- #
# host <-> device plumbing
# --------------------------------------------------------------------------- #
def is_torch(x):
    return type(x).__module__.startswith("torch")


def _values(x):
    """DataFrame / Series -> ndarray (reference: X.values, backend/sglm_ez.py:376-377); a device-resident
    design (sglm_pp.DeviceDesign) -> its CUDA tensor."""
    if type(x).__name__ == "DeviceDesign":
        return x.tensor()
    if hasattr(x, "values") and not is_torch(x) and not isinstance(x, np.ndarray):
        return x.values
    return x


def device_matrix(X):
    """2-D float64 CUDA tensor with unit column stride (rows may be strided: views of a
    larger design matrix are used as they are, no copy)."""
    torch = nat.require_cuda()
    X = _values(X)
    if is_torch(X):
        t = X
        if t.dim() == 1:
            t = t[:, None]
        if t.dtype != torch.float64:
            t = t.to(torch.float64)
        if not t.is_cuda:
            t = t.to("cuda", non_blocking=True)
        if t.dim() != 2:
            raise ValueError(f"Expected 2D array, got {t.dim()}D")
        if t.shape[1] > 0 and t.stride(1) != 1 or (t.shape[0] > 1 and t.stride(0) < t.shape[1]):
            t = t.contiguous()
        return t
    a = np.asarray(X)
    if a.ndim == 1:
        a = a.reshape(-1, 1)
    if a.ndim != 2:
        raise ValueError(f"Expected 2D array, got {a.ndim}D array instead")
    a = np.ascontiguousarray(a, dtype=np.float64)
    if not a.flags.writeable:
        a = a.copy()
    return torch.from_numpy(a).to("cuda")


def device_vector(y):
    torch = nat.require_cuda()
    y = _values(y)
    if is_torch(y):
        t = y.reshape(-1)
        if t.dtype != torch.float64:
            t = t.to(torch.float64)
        if not t.is_cuda:
            t = t.to("cuda", non_blocking=True)
        return t.contiguous()
    a = np.ascontiguousarray(np.asarray(y).reshape(-1), dtype=np.float64)
    if not a.flags.writeable:
        a = a.copy()
    return torch.from_numpy(a).to("cuda")


def row_stride(t):
    return t.stride(0) if t.shape[0] > 1 else max(t.shape[1], 1)


def _empty(shape, dtype=None):
    torch = nat.require_cuda()
    return torch.empty(shape, dtype=dtype or torch.float64, device="cuda")


def _zeros(shape, dtype=None):
    torch = nat.require_cuda()
    return torch.zeros(shape, dtype=dtype or torch.float64, device="cuda")


def _dev(a, dtype):
    torch = nat.require_cuda()
    return torch.from_numpy(np.ascontiguousarray(a, dtype=dtype)).to("cuda")


def _round_up(x, m):
    return (x + m - 1) // m * m


# --------------------------------------------------------------------------- #
# (a1-a3) gather
# --------------------------------------------------------------------------- #
def gather(Xd, col_src, col_shift, fill_value):
    """out[t, c] = Xd[t - col_shift[c], col_src[c]] or fill (sglm_timeshift_f64_ranged)."""
    T, P = Xd.shape
    col_src = np.ascontiguousarray(col_src, dtype=np.int32)
    col_shift = np.ascontiguousarray(col_shift, dtype=np.int32)
    C = int(col_src.shape[0])
    out = _empty((T, C))
    if T == 0 or C == 0:
        return out
    if col_src.min() < 0 or col_src.max() >= P:
        raise IndexError("shift_inx out of bounds for the columns of X")
    both = _dev(np.concatenate([col_src, col_shift]), np.int32)
    call("sglm_timeshift_f64_ranged", ptr(Xd), T, P, row_stride(Xd), ptr(both[:C]), ptr(both[C:]), C,
         int(col_shift.min()), int(col_shift.max()), nat.f64_bits(fill_value), ptr(out), C, stream_ptr())
    return out


class LagRecipe:
    """A lag design that has not been built: base signals on the device + column map + a contiguous row range
    (what `sglm_pp.DeviceDesign` holds after `dropna()`).  Design row t (0-based inside the range), column c is
    base[lo + t - sh[c], src[c]].  The tensor-core statistics are computed from the base signals alone
    (suffstats_tc -> sglm_gram_tc_lag_cells_f64: the 32 GB design of BASELINE configs[2] is neither written nor read);
    everything else asks for `tensor()`, which gathers the design once (cached)."""

    def __init__(self, base, src, sh, lo, hi, fill, cache=None):
        self.base = base
        self.src = np.ascontiguousarray(src, dtype=np.int32)
        self.sh = np.ascontiguousarray(sh, dtype=np.int32)
        self.lo, self.hi, self.fill = int(lo), int(hi), fill
        self._cache = cache

    @property
    def shape(self):
        return (max(self.hi - self.lo, 0), int(self.src.shape[0]))

    def window(self):
        """(u0, n_u, off): rows [u0, u0 + n_u) of the base signals hold everything the design reads, design row t of
        column c is window row t + off[c]; None when a column reads outside the base signals (fill values)."""
        if self.src.shape[0] == 0 or self.hi <= self.lo:
            return None
        u0, u1 = self.lo - int(self.sh.max()), self.hi - int(self.sh.min())
        if u0 < 0 or u1 > int(self.base.shape[0]):
            return None
        return u0, u1 - u0, np.ascontiguousarray(self.lo - self.sh - u0, dtype=np.int32)

    def tensor(self):
        if self._cache is None:
            # only the base rows the range reads (lag halo included): a row slice of a long session (one rank of a
            # row-sharded grid) costs its own rows, not the whole session
            sh_max, sh_min = (int(self.sh.max()), int(self.sh.min())) if self.sh.size else (0, 0)
            a = max(0, min(self.lo, self.lo - sh_max))
            b = min(int(self.base.shape[0]), max(self.hi, self.hi - sh_min))
            if b <= a:
                a = b = min(max(self.lo, 0), int(self.base.shape[0]))
            self._cache = gather(self.base[a:b], self.src, self.sh, self.fill)[self.lo - a:self.hi - a]
        return self._cache


def device_design(X):
    """device_matrix(X), except that a device-resident lag design with a contiguous row range stays a recipe
    (LagRecipe) — the Gaussian CV grid computes its statistics from the base signals."""
    if type(X).__name__ == "DeviceDesign":
        r = X.lag_recipe()
        if r is not None:
            return r
    return device_matrix(X)


def _lag_analysis(Xr, Yd, win, all_reduce=None):
    """Column analysis of a lag design from its base signals: exponents / digit planes of [base | 1] over the window
    (every lag column inherits those of its base signal) and of [Y | 1].  Returns device colE, colS [n_aug],
    baseE, baseS [P + 1] and a device flag tensor (NaN / inf seen)."""
    torch = nat.require_cuda()
    u0, n_u, _ = win
    P = int(Xr.base.shape[1])
    n_y = Yd.shape[1]
    T = Xr.shape[0]
    bw = Xr.base[u0:u0 + n_u]
    cm_b = torch.empty(P + 1, dtype=torch.int64, device="cuda")
    ls_b = torch.empty(P + 1, dtype=torch.int32, device="cuda")
    cm_y = torch.empty(n_y + 1, dtype=torch.int64, device="cuda")
    ls_y = torch.empty(n_y + 1, dtype=torch.int32, device="cuda")
    call("sglm_gram_tc_colstats_f64", ptr(bw), row_stride(bw), None, 0, 0, n_u, P, ptr(cm_b), ptr(ls_b), stream_ptr())
    call("sglm_gram_tc_colstats_f64", None, 0, ptr(Yd), row_stride(Yd), n_y, T, 0, ptr(cm_y), ptr(ls_y), stream_ptr())
    if all_reduce is not None:
        cm = torch.cat([cm_b, cm_y]); ls = torch.cat([ls_b, ls_y])
        all_reduce(cm, "max"); all_reduce(ls, "min")
        cm_b, cm_y, ls_b, ls_y = cm[:P + 1].contiguous(), cm[P + 1:].contiguous(), ls[:P + 1].contiguous(), ls[P + 1:].contiguous()
    bE = torch.empty(P + 1, dtype=torch.int32, device="cuda")
    yE = torch.empty(n_y + 1, dtype=torch.int32, device="cuda")
    flags = torch.empty(2, dtype=torch.int32, device="cuda")
    call("sglm_gram_tc_exponents", ptr(cm_b), P + 1, 8, ptr(bE), ptr(ls_b), ptr(flags[0:]), stream_ptr())
    call("sglm_gram_tc_exponents", ptr(cm_y), n_y + 1, 8, ptr(yE), ptr(ls_y), ptr(flags[1:]), stream_ptr())
    src_t = _dev(Xr.src, np.int64)
    colE = torch.cat([bE.index_select(0, src_t), yE]).contiguous()
    colS = torch.cat([ls_b.index_select(0, src_t), ls_y]).contiguous()
    return colE, colS, bE, ls_b, flags


# --------------------------------------------------------------------------- #
# sufficient statistics
# --------------------------------------------------------------------------- #
def index_counts(idx, T):
    """Row multiplicities of an index list (X[idx, :] semantics incl. repeats / negatives)."""
    torch = nat.require_cuda()
    counts = _zeros((T,))
    if is_torch(idx):
        it = idx.to(device="cuda", dtype=torch.int64).contiguous()
    else:
        a = np.asarray(idx)
        if a.dtype == bool:
            a = np.flatnonzero(a)
        it = _dev(a.reshape(-1), np.int64)
    if it.numel():
        call("sglm_index_counts_f64", ptr(it), it.numel(), ptr(counts), T, stream_ptr())
    return counts


def roll_vector(yd, shift):
    """np.roll(y, shift) on the device (backend/sglm_cv.py:95-96)."""
    out = _empty((yd.numel(),))
    call("sglm_roll_f64", ptr(yd), yd.numel(), int(shift), ptr(out), stream_ptr())
    return out


def sorted_unique_rows(idx_t, T):
    """Ascending, duplicate-free positions of an index list (CUDA int64, values in [0, T)) without a sort: a row
    mask (duplicates detected while setting it) followed by an ordered compaction.  Returns a tensor SHORTER than
    the input when the list repeats rows."""
    torch = nat.require_cuda()
    mask = torch.empty((T + 3) // 4 * 4 + 4, dtype=torch.uint8, device="cuda")
    flags = torch.empty(4, dtype=torch.int64, device="cuda")            # [0] duplicate flag (int32 view)
    call("sglm_index_mask_u8", ptr(idx_t), idx_t.numel(), ptr(mask), T, ptr(flags), stream_ptr())
    dup = int(flags.view(torch.int32)[0].item())
    n = int(idx_t.numel())
    if dup:
        return idx_t[:max(n - 1, 0)]
    rows = torch.empty(n, dtype=torch.int64, device="cuda")
    wb = nat.lib().sglm_mask_compact_workspace_bytes(T)
    ws = torch.empty((wb + 7) // 8, dtype=torch.int64, device="cuda")
    call("sglm_mask_compact_rows", ptr(mask), T, ptr(rows), ptr(ws), ws.numel() * 8, stream_ptr())
    return rows


def suffstats(Xd, Yd, W=None, rows_hint=None):
    """G[s] = Z' diag(W[s]) Z with Z = [X | Y | 1].  W: [n_sets, T] tensor or None (one
    unit-weight set).  Returns G [n_sets, n_aug, ldg] (full symmetric)."""
    T, C = Xd.shape
    n_y = Yd.shape[1]
    n_sets = 1 if W is None else W.shape[0]
    n_aug = C + n_y + 1
    ldg = _round_up(n_aug, 8)
    G = _zeros((n_sets, n_aug, ldg))       # padding columns stay zero
    n_tiles = max(1, (T + 15) // 16)
    n_pairs = ((n_aug + 127) // 128) * (((n_aug + 127) // 128) + 1) // 2
    rows = np.asarray(rows_hint if rows_hint is not None else [T] * n_sets, dtype=np.float64)
    rows = np.maximum(rows, 1.0)
    ks = np.maximum(1, np.minimum(np.maximum(1, (rows / 16).astype(np.int64) // 64),
                                  np.rint(_SM_TARGET_ITEMS * rows / rows.sum() / n_pairs).astype(np.int64)))
    ks = np.ascontiguousarray(np.minimum(ks, n_tiles), dtype=np.int32)
    ks_p = ks.ctypes.data_as(ctypes.c_void_p)
    ws_bytes = nat.lib().sglm_suffstats_workspace_bytes(T, C, n_y, n_sets, ks_p)
    if ws_bytes == 0:
        raise nat.SglmNativeError("suffstats: invalid plan: " + nat.lib().sglm_last_error().decode())
    torch = nat.require_cuda()
    ws = torch.empty((ws_bytes + 255) // 256 * 32, dtype=torch.float64, device="cuda")
    call("sglm_suffstats_f64", ptr(Xd), row_stride(Xd), ptr(Yd), row_stride(Yd), n_y, T, C,
         ptr(W), (W.stride(0) if W is not None else 0), n_sets, ks_p, ptr(G), ldg, ptr(ws), ws.numel() * 8,
         stream_ptr())
    return G


def suffstats_tc(Xd, Yd, set_rows, check_gemm=False):
    """Tensor-core Gram (tcgen05 int8 digit planes, exact integer accumulation, fp64
    recombination): same output as `suffstats` for 0/1 row sets.
    set_rows: list with one entry per set — None (all rows) or a sorted, duplicate-free int64
    CUDA tensor of row indices.  Returns G [n_sets, n_aug, ldg]."""
    torch = nat.require_cuda()
    lag = win = None
    if isinstance(Xd, LagRecipe):
        win = None if check_gemm else Xd.window()
        if win is None:
            Xd = Xd.tensor()
        else:
            lag = Xd
    T, C = Xd.shape
    n_y = Yd.shape[1]
    n_aug = C + n_y + 1
    n_sets = len(set_rows)
    ldg = _round_up(n_aug, 8)
    if lag is not None:
        colE, colS, baseE, baseS, flags = _lag_analysis(lag, Yd, win)
        host = torch.cat([colS, baseS, flags]).cpu().numpy()
        if host[-2:].any():
            raise ValueError("Input contains NaN, infinity or a value too large for dtype('float64').")
        colS_h = np.ascontiguousarray(host[:n_aug], dtype=np.int32)
        baseS_h = np.ascontiguousarray(host[n_aug:-2], dtype=np.int32)
    else:
        colE = torch.empty(n_aug, dtype=torch.int32, device="cuda")
        colS = torch.empty(n_aug, dtype=torch.int32, device="cuda")
        scratch = torch.empty(n_aug, dtype=torch.int64, device="cuda")
        flag = torch.empty(1, dtype=torch.int32, device="cuda")
        call("sglm_gram_tc_analyze_f64", ptr(Xd), row_stride(Xd), ptr(Yd), row_stride(Yd), n_y, T, C, ptr(colE),
             ptr(colS), ptr(scratch), ptr(flag), stream_ptr())
        host = torch.cat([colS, flag]).cpu().numpy()
        if host[-1] != 0:
            raise ValueError("Input contains NaN, infinity or a value too large for dtype('float64').")
        colS_h = np.ascontiguousarray(host[:-1], dtype=np.int32)
    cells = None if TC_CELLS is False else _row_cells(set_rows, T)
    if cells is None:
        lists = [torch.arange(T, dtype=torch.int64, device="cuda") if r is None else r.to(torch.int64) for r in set_rows]
        member = None
    else:
        lists, member = cells
    n_lists = len(lists)
    sizes = np.ascontiguousarray([int(r.numel()) for r in lists], dtype=np.int64)
    parts = []
    for body, n in zip(lists, sizes):
        pad = (-int(n)) % 128
        parts.append(body)
        if pad:
            parts.append(torch.full((pad,), -1, dtype=torch.int64, device="cuda"))
    rows = torch.cat(parts) if parts else torch.empty(0, dtype=torch.int64, device="cuda")
    if rows.numel() == 0:
        rows = torch.full((128,), -1, dtype=torch.int64, device="cuda")
    colS_p, sizes_p = colS_h.ctypes.data_as(ctypes.c_void_p), sizes.ctypes.data_as(ctypes.c_void_p)
    if lag is not None:
        u0, n_u, off_h = win
        P = int(lag.base.shape[1])
        ws_bytes = nat.lib().sglm_gram_tc_lag_workspace_bytes(n_aug, colS_p, n_lists, sizes_p, 0 if member is None else n_sets, P,
                                                              baseS_h.ctypes.data_as(ctypes.c_void_p), n_u)
    elif member is None:
        ws_bytes = nat.lib().sglm_gram_tc_workspace_bytes(n_aug, colS_p, n_lists, sizes_p)
    else:
        ws_bytes = nat.lib().sglm_gram_tc_cells_workspace_bytes(n_aug, colS_p, n_lists, sizes_p, n_sets)
    if ws_bytes == 0:
        raise nat.SglmNativeError("gram_tc: invalid plan")
    info = np.zeros(4, dtype=np.int64)
    nat.lib().sglm_gram_tc_plan_info(n_aug, colS_p, n_lists, sizes_p, info.ctypes.data_as(ctypes.c_void_p))
    nat.last_tc_plan = dict(S=int(info[0]), n_pos=int(info[1]), tiles=int(info[2]), k_parts=int(info[3]),
                            planes=int(colS_h.sum()), n_aug=n_aug, row_lists=n_lists, cells=member is not None,
                            lag=lag is not None)
    raw = torch.empty(ws_bytes + 1024, dtype=torch.uint8, device="cuda")
    off = (-raw.data_ptr()) % 1024
    G = _zeros((n_sets, n_aug, ldg))
    if lag is not None:
        bw = lag.base[u0:u0 + n_u]
        desc = nat.LagDesignStruct(bw.data_ptr(), row_stride(bw), n_u, P, lag.src.ctypes.data, off_h.ctypes.data,
                                   baseE.data_ptr(), baseS.data_ptr(), baseS_h.ctypes.data)
        member_p = None if member is None else np.ascontiguousarray(member, dtype=np.int32)
        call("sglm_gram_tc_lag_cells_f64", ctypes.byref(desc), ptr(Yd), row_stride(Yd), n_y, T, C, ptr(colE), ptr(colS), colS_p,
             n_lists, sizes_p, ptr(rows), 0 if member is None else n_sets,
             None if member_p is None else member_p.ctypes.data_as(ctypes.c_void_p), ptr(G), ldg,
             ctypes.c_void_p(raw.data_ptr() + off), ws_bytes, 0, stream_ptr())
    elif member is None:
        call("sglm_gram_tc_f64", ptr(Xd), row_stride(Xd), ptr(Yd), row_stride(Yd), n_y, T, C, ptr(colE), ptr(colS),
             colS_p, n_lists, sizes_p, ptr(rows), ptr(G), ldg, ctypes.c_void_p(raw.data_ptr() + off), ws_bytes,
             int(bool(check_gemm)), stream_ptr())
    else:
        member = np.ascontiguousarray(member, dtype=np.int32)
        call("sglm_gram_tc_cells_f64", ptr(Xd), row_stride(Xd), ptr(Yd), row_stride(Yd), n_y, T, C, ptr(colE),
             ptr(colS), colS_p, n_lists, sizes_p, ptr(rows), n_sets, member.ctypes.data_as(ctypes.c_void_p), ptr(G), ldg,
             ctypes.c_void_p(raw.data_ptr() + off), ws_bytes, int(bool(check_gemm)), stream_ptr())
    return G, colS_h


def suffstats_tc_sharded(Xd, Yd, set_rows, all_reduce):
    """Row-sharded tensor-core Gram: this process holds a SLICE of the rows (Xd, Yd, set_rows in local row
    numbers); `all_reduce(tensor, op)` combines a CUDA tensor over the processes in place (op in "max", "min",
    "sum").  Three small collectives: column maxima (int64 max) and lowest set bits (int32 min) so that every rank
    cuts the same digit planes, then the int64 plane Grams of the row sets (sum — exact integer arithmetic, so the
    result has the bits of the one-GPU computation).  Returns G [n_sets, n_aug, ldg], identical on every rank."""
    torch = nat.require_cuda()
    lag = win = None
    if isinstance(Xd, LagRecipe):
        # every rank must take the same path: a rank whose slice reads outside the base signals (fill values) makes all
        # ranks build their slices
        win = Xd.window()
        ok = torch.tensor([0 if win is None else 1], dtype=torch.int32, device="cuda")
        all_reduce(ok, "min")
        if int(ok.item()) == 0:
            win = None
            Xd = Xd.tensor()
        else:
            lag = Xd
    T, C = Xd.shape
    n_y = Yd.shape[1]
    n_aug = C + n_y + 1
    n_sets = len(set_rows)
    ldg = _round_up(n_aug, 8)
    if lag is not None:
        # the analysis of the base signals, combined over the ranks: the union of the ranks' windows is the window of
        # the one-GPU computation, so the digit planes (and the summed int64 plane Grams) are the same bits
        colE, colS, baseE, baseS, flags = _lag_analysis(lag, Yd, win, all_reduce)
        host = torch.cat([colS, baseS, flags]).cpu().numpy()
        if host[-2:].any():
            raise ValueError("Input contains NaN, infinity or a value too large for dtype('float64').")
        colS_h = np.ascontiguousarray(host[:n_aug], dtype=np.int32)
        baseS_h = np.ascontiguousarray(host[n_aug:-2], dtype=np.int32)
    else:
        colmax = torch.empty(n_aug, dtype=torch.int64, device="cuda")
        colS = torch.empty(n_aug, dtype=torch.int32, device="cuda")
        colE = torch.empty(n_aug, dtype=torch.int32, device="cuda")
        flag = torch.empty(1, dtype=torch.int32, device="cuda")
        call("sglm_gram_tc_colstats_f64", ptr(Xd), row_stride(Xd), ptr(Yd), row_stride(Yd), n_y, T, C, ptr(colmax), ptr(colS),
             stream_ptr())
        all_reduce(colmax, "max")            # bits of non-negative doubles order like integers; the NaN pattern wins
        all_reduce(colS, "min")
        call("sglm_gram_tc_exponents", ptr(colmax), n_aug, 8, ptr(colE), ptr(colS), ptr(flag), stream_ptr())
        host = torch.cat([colS, flag]).cpu().numpy()
        if host[-1] != 0:
            raise ValueError("Input contains NaN, infinity or a value too large for dtype('float64').")
        colS_h = np.ascontiguousarray(host[:-1], dtype=np.int32)
    cells = _row_cells(set_rows, T)
    if cells is None:                    # no overlap among this rank's rows: every set is its own cell
        lists = [torch.arange(T, dtype=torch.int64, device="cuda") if r is None else r.to(torch.int64) for r in set_rows]
        member = np.eye(n_sets, dtype=np.int32)
    else:
        lists, member = cells
    n_lists = len(lists)
    sizes = np.ascontiguousarray([int(r.numel()) for r in lists], dtype=np.int64)
    parts = []
    for body, n in zip(lists, sizes):
        parts.append(body)
        pad = (-int(n)) % 128
        if pad:
            parts.append(torch.full((pad,), -1, dtype=torch.int64, device="cuda"))
    rows = torch.cat(parts) if parts else torch.empty(0, dtype=torch.int64, device="cuda")
    if rows.numel() == 0:
        rows = torch.full((128,), -1, dtype=torch.int64, device="cuda")
    colS_p, sizes_p = colS_h.ctypes.data_as(ctypes.c_void_p), sizes.ctypes.data_as(ctypes.c_void_p)
    if lag is not None:
        u0, n_u, off_h = win
        P = int(lag.base.shape[1])
        ws_bytes = nat.lib().sglm_gram_tc_lag_workspace_bytes(n_aug, colS_p, n_lists, sizes_p, n_sets, P,
                                                              baseS_h.ctypes.data_as(ctypes.c_void_p), n_u)
    else:
        ws_bytes = nat.lib().sglm_gram_tc_cells_workspace_bytes(n_aug, colS_p, n_lists, sizes_p, n_sets)
    if ws_bytes == 0:
        raise nat.SglmNativeError("gram_tc: invalid plan")
    off_b, size_b = ctypes.c_uint64(0), ctypes.c_uint64(0)
    if nat.lib().sglm_gram_tc_cells_sgout(n_aug, colS_p, n_lists, sizes_p, n_sets, ctypes.byref(off_b), ctypes.byref(size_b)) != 0:
        raise nat.SglmNativeError("gram_tc: " + nat.lib().sglm_last_error().decode())
    info = np.zeros(4, dtype=np.int64)
    nat.lib().sglm_gram_tc_plan_info(n_aug, colS_p, n_lists, sizes_p, info.ctypes.data_as(ctypes.c_void_p))
    nat.last_tc_plan = dict(S=int(info[0]), n_pos=int(info[1]), tiles=int(info[2]), k_parts=int(info[3]),
                            planes=int(colS_h.sum()), n_aug=n_aug, row_lists=n_lists, cells=cells is not None, sharded=True,
                            lag=lag is not None)
    raw = torch.empty(ws_bytes + 1024, dtype=torch.uint8, device="cuda")
    off = (-raw.data_ptr()) % 1024
    ws_p = ctypes.c_void_p(raw.data_ptr() + off)
    member = np.ascontiguousarray(member, dtype=np.int32)
    if lag is not None:
        bw = lag.base[u0:u0 + n_u]
        desc = nat.LagDesignStruct(bw.data_ptr(), row_stride(bw), n_u, P, lag.src.ctypes.data, off_h.ctypes.data,
                                   baseE.data_ptr(), baseS.data_ptr(), baseS_h.ctypes.data)
        call("sglm_gram_tc_lag_cells_f64", ctypes.byref(desc), ptr(Yd), row_stride(Yd), n_y, T, C, ptr(colE), ptr(colS), colS_p,
             n_lists, sizes_p, ptr(rows), n_sets, member.ctypes.data_as(ctypes.c_void_p), None, ldg, ws_p, ws_bytes, 1,
             stream_ptr())
    else:
        call("sglm_gram_tc_cells_partial_f64", ptr(Xd), row_stride(Xd), ptr(Yd), row_stride(Yd), n_y, T, C, ptr(colE),
             ptr(colS), colS_p, n_lists, sizes_p, ptr(rows), n_sets, member.ctypes.data_as(ctypes.c_void_p), ws_p, ws_bytes,
             stream_ptr())
    sg = raw[off + off_b.value: off + off_b.value + size_b.value].view(torch.int64)
    all_reduce(sg, "sum")
    G = _zeros((n_sets, n_aug, ldg))
    call("sglm_gram_tc_cells_combine_f64", C, n_y, ptr(colE), ptr(colS), colS_p, n_lists, sizes_p, n_sets, ptr(G), ldg,
         ws_p, ws_bytes, stream_ptr())
    return G


TC_CELLS = None      # False: one GEMM pass per row set (no cell decomposition); None: decompose when it pays
_MAX_CELLS = 64


def _row_cells(set_rows, T):
    """Disjoint cells of the partition of the rows induced by overlapping row sets.
    set_rows: None (all rows) or sorted duplicate-free int64 CUDA tensors.  Returns
    ([rows of cell c], member[n_sets][n_cells]) or None when the decomposition does not pay
    (no overlap, too many sets or cells).  The full data of a CV grid contain every test fold and
    random folds (GroupShuffleSplit, backend/sglm_pp.py:262-263) intersect: the cells are visited
    once by the GEMM, the sets are integer sums of cell Grams."""
    torch = nat.require_cuda()
    listed = [i for i, r in enumerate(set_rows) if r is not None]
    if not listed or len(listed) > 60 or len(set_rows) < 2:
        return None
    any_all = len(listed) < len(set_rows)
    # row signatures (bit b = row is in listed set b), distinct signatures = cells: a 256-slot hash table on the
    # device, one read-back of the table (keys + counts), then one ordered compaction per cell — no sort
    sig = torch.zeros(max(T, 1), dtype=torch.int64, device="cuda")
    for bit, i in enumerate(listed):
        r = set_rows[i].to(torch.int64)
        call("sglm_rows_or_bit_u64", ptr(r), r.numel(), bit, ptr(sig), T, stream_ptr())
    cell_of = torch.empty(max(T, 1), dtype=torch.uint8, device="cuda")
    table = torch.empty(513 + 1, dtype=torch.int64, device="cuda")
    call("sglm_cells_from_signatures", ptr(sig), T, ptr(cell_of), ptr(table), stream_ptr())
    th = table.cpu().numpy()
    keys_h, counts_h, flags = th[:256], th[256:512], th[512:513].view(np.int32)
    if flags[1] != 0:
        return None
    slots = [int(sl) for sl in np.flatnonzero(counts_h > 0)]
    slots.sort(key=lambda sl: int(keys_h[sl]) & 0xFFFFFFFFFFFFFFFF)           # ascending signature: a fixed cell order
    if len(slots) > _MAX_CELLS + 1:
        return None
    total_listed = sum(int(set_rows[i].numel()) for i in listed) + (T if any_all else 0) * (len(set_rows) - len(listed))
    cell_rows = sum(int(counts_h[sl]) for sl in slots if any_all or keys_h[sl] != 0)
    if cell_rows >= total_listed:             # disjoint sets: nothing to share
        return None
    lists, member_cols = [], []
    bit_of = {i: b for b, i in enumerate(listed)}
    wb = nat.lib().sglm_mask_compact_workspace_bytes(T)
    ws = torch.empty((wb + 7) // 8, dtype=torch.int64, device="cuda")
    for sl in slots:
        u = int(keys_h[sl])
        if u == 0 and not any_all:
            continue
        rows_c = torch.empty(int(counts_h[sl]), dtype=torch.int64, device="cuda")
        call("sglm_match_compact_rows", ptr(cell_of), T, sl, ptr(rows_c), ptr(ws), ws.numel() * 8, stream_ptr())
        lists.append(rows_c)
        member_cols.append([1 if r is None else int((u >> bit_of[i]) & 1) for i, r in enumerate(set_rows)])
    member = np.array(member_cols, dtype=np.int32).T          # [n_sets][n_cells]
    return lists, member


class Problem:
    """Centred problem (Qc, qc, yyc, xbar, ybar, n) of one (row set, y column, intercept)."""
    __slots__ = ("Qc", "qc", "xbar", "diag", "scal", "ldq", "fit_intercept", "y_col", "n", "ybar", "yyc", "sy")


def center(A_plus, A_minus, C, n_y, y_col, fit_intercept, n_rows=None):
    """n_rows: number of rows of the set when the caller knows it (then no device read-back is
    needed before the solvers: everything else about the problem stays on the device)."""
    ldg = A_plus.stride(0)
    ldq = _round_up(C, 8)
    p = Problem()
    p.Qc = _empty((C, ldq))
    p.qc = _empty((C,))
    p.xbar = _empty((C,))
    p.diag = _empty((C,))
    p.scal = _empty((4,))
    p.ldq, p.fit_intercept, p.y_col = ldq, bool(fit_intercept), y_col
    p.n = float(n_rows) if n_rows is not None else None
    call("sglm_center_stats_f64", ptr(A_plus), ptr(A_minus), ldg, C, n_y, y_col, int(bool(fit_intercept)),
         ptr(p.Qc), ldq, ptr(p.qc), ptr(p.xbar), ptr(p.diag), ptr(p.scal), stream_ptr())
    return p


def fetch_scalars(problems):
    """One D2H copy for the (yyc, n, ybar, sum_y) of all problems."""
    torch = nat.require_cuda()
    if not problems:
        return
    host = torch.stack([p.scal for p in problems]).cpu().numpy()
    for p, s in zip(problems, host):
        p.yyc, p.n, p.ybar, p.sy = (float(v) for v in s)


# --------------------------------------------------------------------------- #
# batched solvers
# --------------------------------------------------------------------------- #
class ModelSpec:
    """One fit of the grid: which problem, which penalty."""
    __slots__ = ("problem", "kind", "alpha", "l1_ratio", "max_iter", "tol", "coef_init")

    def __init__(self, problem, kind, alpha=1.0, l1_ratio=0.5, max_iter=1000, tol=1e-4, coef_init=None):
        self.problem, self.kind = problem, kind
        self.alpha, self.l1_ratio = float(alpha), float(l1_ratio)
        self.max_iter, self.tol, self.coef_init = int(max_iter), float(tol), coef_init


WARM_START_PATHS = False     # opt-in (non-reference) mode, see solve_models


def _warm_paths():
    import os
    return WARM_START_PATHS or os.environ.get("SGLM_WARM_PATH", "0") == "1"


CD_DEBUG_TIMER = 0      # diagnostics: which timer of the cluster kernel lands in info[:, 5] (0 register phase, 1 waits, 2 publish, 3 look-ahead)
CD_GROUP, CD_CLUSTER = None, None     # override of (models per cluster, CTAs per cluster); 0 = first-generation kernel


CD_PLAN = None      # override of the launch plan, e.g. "4x2@0.2,4x1" (see _cd_plan)
CD_COLLECT_STATS = False   # bench.py: keep per-part device statistics of the coordinate-descent launches
cd_parts_log = []          # [{shape (M, K), slots (r0, r1), group_stats [n_groups, 2] | None, info [n_slots, 6]}]


def cd_stats():
    """Summary of the logged coordinate-descent parts (synchronises): rows of Q loaded through L2 (a moved row
    once per cluster group; once per model in the per-model kernel), coordinate updates, the longest chain of
    coordinate blocks one model walked.  Clears the log."""
    out = []
    for part in cd_parts_log:
        r0, r1 = part["slots"]
        info = part["info"][r0:r1].cpu().numpy()
        rows = float(part["group_stats"][:, 0].sum().item()) if part["group_stats"] is not None else float(info[:, 3].sum())
        out.append(dict(shape="%dx%d" % part["shape"], models=r1 - r0, row_updates=float(info[:, 3].sum()),
                        rows_loaded=rows, max_blocks_one_model=float(info[:, 4].max()) if r1 > r0 else 0.0,
                        max_sweeps=float(info[:, 2].max()) if r1 > r0 else 0.0,
                        register_phase_share_heaviest=float(info[int(np.argmax(info[:, 4])), 5]) if r1 > r0 else 0.0))
    cd_parts_log.clear()
    return out
_SIDE_STREAMS = {}


def _side_stream(i):
    torch = nat.require_cuda()
    key = (torch.cuda.current_device(), i)
    if key not in _SIDE_STREAMS:
        _SIDE_STREAMS[key] = torch.cuda.Stream()
    return _SIDE_STREAMS[key]


def _cd_shape_ok(g, k, C):
    if g <= 0 or k <= 0:
        return 0, 0
    while k > 1 and (C + 31) // 32 < 2 * k:
        k //= 2
    if g == 8 and k < 2:
        g = 4                 # groups of 8 exist for clusters of 2+ CTAs only
    if not nat.lib().sglm_enet_cd_cluster_supported(g, k):
        raise nat.SglmNativeError(f"coordinate descent: unsupported (group, cluster) = ({g}, {k})")
    # very wide designs: a CTA's column slice (w and Qw of every model of the group) must fit in shared memory
    # — widen the cluster, then shrink the group, else fall back to one CTA per model
    limit = 227 * 1024
    while nat.lib().sglm_enet_cd_cluster_smem_bytes(g, k, C) > limit:
        if k < 8 and (C + 31) // 32 >= 4 * k:
            k *= 2
        elif g > 1:
            g //= 2
        else:
            return 0, 0
    return g, k


def _cd_plan(C, n_models, n_probs=1):
    """Parts of the coordinate-descent launch: [(first slot, end slot, group size M, cluster size K)] over
    the cost-ordered model list (heaviest first).  Plan text: comma-separated `MxK[@fraction]` or `MxK[#count]`;
    a part takes `fraction` of the models / `count` models (the last part takes the rest); `0x0` is the
    first-generation one-CTA-per-model kernel.  CD_GROUP / CD_CLUSTER (or SGLM_CD_GROUP / SGLM_CD_CLUSTER) give a
    one-part plan."""
    import os
    g = CD_GROUP if CD_GROUP is not None else os.environ.get("SGLM_CD_GROUP")
    k = CD_CLUSTER if CD_CLUSTER is not None else os.environ.get("SGLM_CD_CLUSTER")
    text = CD_PLAN if CD_PLAN is not None else os.environ.get("SGLM_CD_PLAN")
    if g is not None or k is not None:
        text = f"{int(1 if g is None else g)}x{int(1 if k is None else k)}"
    if text is None:
        text = _CD_DEFAULT_PLAN(C, n_models, n_probs)
    parts, r0 = [], 0
    items = [t for t in text.split(",") if t]
    for n, item in enumerate(items):
        shape, sep, frac = item.partition("@")
        if not sep:
            shape, sep, count = item.partition("#")
            frac = ""
        else:
            count = ""
        gg, kk = (int(v) for v in shape.split("x"))
        if n == len(items) - 1 or not (frac or count):
            r1 = n_models
        elif count:
            r1 = min(n_models, r0 + int(count))
        else:
            r1 = min(n_models, r0 + int(round(float(frac) * n_models)))
        gg, kk = _cd_shape_ok(gg, kk, C)
        parts.append((r0, r1, gg, kk))
        r0 = r1
    return parts


def _CD_DEFAULT_PLAN(C, n_models, n_probs=1):
    # wide designs: the heaviest 30 % of the cost-ordered grid as groups of M models of one fold on K-CTA clusters,
    # the light rest concurrently on the one-CTA-per-model kernel.  A model is a serial chain of 32-coordinate
    # blocks; measured per block for the heaviest model (profiles/r2_cd_experiments.txt): 6.1 us on (4,2), 4.0 us
    # on (4,4), 3.4 us on (2,4), 3.2 us on (1,8) — wider clusters shorten the chain but need more SMs per model.  The
    # block counts fall quickly with the rank in the cost order, so only the HEAD of the order (the heaviest group of
    # every problem) is chain-critical and gets the widest shape the GPU can afford; the shapes behind it follow the SMs
    # that are left (experiments log sections 7 and 15):
    #   a whole grid (>= ~800 models):  head on (4,4), rest of the heavy part on (4,2)         1500 models: 354 -> 288 ms
    #   a share of a grid (one of 2-4 GPUs): head on (2,4), then (4,4) while SMs last, then (4,2)  750: 231 -> 204, 375: 208 -> 180
    #   a small share (one of 8 GPUs):  one model per problem on (1,8), the rest on (2,4)      188: 173 -> 163
    # A handful of models (a single GLM.fit) leaves the GPU idle anyway: each model gets a 4-CTA cluster
    # (config 1: CD 5.6 -> 4.3 ms).  Narrow designs keep one CTA per model.
    if C > 1024 and n_models >= 16:
        P = max(1, n_probs)
        heavy = int(round(0.3 * n_models))
        sms = 148
        if n_models <= 250 and P <= heavy and 8 * P <= sms:
            rest = heavy - P
            return f"1x8#{P}," + (f"2x4#{rest}," if rest > 0 else "") + "0x0"
        if n_models <= 800 and 4 * P <= heavy and 8 * P <= sms:
            head = 4 * P                                   # groups of 2 on 4 CTAs: 2 CTAs per model
            rest = heavy - head
            left = int(1.15 * sms) - 2 * head              # CTAs the GPU can still hold at once (slightly oversubscribed)
            n44 = max(0, min(rest, 2 * left - rest))       # (4,4): 1 CTA per model, (4,2): half a CTA per model
            n44 = (n44 + 2 * P) // (4 * P) * (4 * P) if n44 < rest else rest
            n44 = min(n44, rest)
            n42 = rest - n44
            return (f"2x4#{head}," + (f"4x4#{n44}," if n44 > 0 else "") + (f"4x2#{n42}," if n42 > 0 else "") + "0x0")
        head = 4 * P
        if head <= 0.1 * n_models:
            return f"4x4#{head},4x2#{heavy - head},0x0"
        return "4x2@0.3,0x0"
    if C >= 256 and n_models <= 8:
        return "1x4"
    return "0x0"


def solve_models(models, C, do_screening=True):
    """Solve every model; returns (W [M, ldw] device, info [M,6] host, status list).
    ElasticNet/Lasso: one batched coordinate-descent launch.  Ridge/OLS: one Cholesky
    launch per problem (one CTA per alpha).

    Reference semantics = cold start for every model (backend/sglm_cv.py:122 passes
    beta_=None), which is what runs by default.  With `WARM_START_PATHS` (or
    SGLM_WARM_PATH=1) the models of one (problem, l1_ratio) are chained along decreasing
    alpha, each starting from its predecessor's solution (a regularisation path, one launch
    per path position): far fewer sweeps, same optimum — identical to the cold-start result
    only up to the solver tolerance, so it is NOT the parity mode."""
    torch = nat.require_cuda()
    M = len(models)
    ldw = _round_up(C, 2)
    W = _zeros((M, ldw))
    info = np.zeros((M, 6))
    status = np.zeros(M, dtype=np.int64)
    cd = [i for i, m in enumerate(models) if m.kind in ("lasso", "enet")]
    if cd:
        probs, pidx = [], {}
        for i in cd:
            p = models[i].problem
            if id(p) not in pidx:
                pidx[id(p)] = len(probs)
                probs.append(p)
        warm_paths = _warm_paths() and all(models[i].coef_init is None for i in cd)
        levels = None
        if warm_paths:
            paths = {}
            for i in cd:
                m = models[i]
                paths.setdefault((pidx[id(m.problem)], m.l1_ratio, m.tol, m.max_iter), []).append(i)
            for key in paths:
                paths[key].sort(key=lambda i: -models[i].alpha)
            depth = max(len(v) for v in paths.values())
            slots, pred, levels = [], [], []
            pos_of = {}
            for k in range(depth):
                start = len(slots)
                for key, v in paths.items():
                    if k < len(v):
                        pos_of[v[k]] = len(slots)
                        slots.append(v[k])
                        pred.append(pos_of[v[k - 1]] if k > 0 else -1)
                levels.append((start, len(slots)))
            cd = list(slots)
        else:
            # longest-running (weakest penalty) models first so that the tail of the launch is short
            cd.sort(key=lambda i: (models[i].alpha * max(models[i].l1_ratio, 1e-3)))
            slots = list(cd)
        slot_prob = [pidx[id(models[i].problem)] for i in cd]
        n_slots = len(slots)
        ldq = probs[0].ldq
        Qp = _dev(np.array([p.Qc.data_ptr() for p in probs], dtype=np.uint64).view(np.int64), np.int64)
        qp = _dev(np.array([p.qc.data_ptr() for p in probs], dtype=np.uint64).view(np.int64), np.int64)
        dp = _dev(np.array([p.diag.data_ptr() for p in probs], dtype=np.uint64).view(np.int64), np.int64)
        yy = torch.stack([p.scal for p in probs])[:, 0].contiguous()       # yyc, stays on the device
        warm = any(models[i].coef_init is not None for i in cd)
        mget = lambda i, f, pad: (f(models[i]) if i >= 0 else pad)
        l1 = [mget(i, lambda m: m.alpha * m.l1_ratio * m.problem.n, 1.0) for i in slots]
        l2 = [mget(i, lambda m: m.alpha * (1.0 - m.l1_ratio) * m.problem.n, 1.0) for i in slots]
        tl = [mget(i, lambda m: m.tol, 1.0) for i in slots]
        pack_f = _dev(np.array([l1, l2, tl], dtype=np.float64), np.float64)
        pack_i = _dev(np.array([slot_prob, [mget(i, lambda m: m.max_iter, 0) for i in slots]], dtype=np.int32), np.int32)
        Wcd = _zeros((n_slots, ldw))
        if warm:
            init = np.zeros((n_slots, ldw))
            for r, i in enumerate(slots):
                if i >= 0 and models[i].coef_init is not None:
                    init[r, :C] = np.asarray(models[i].coef_init, dtype=np.float64).reshape(-1)
            Wcd.copy_(torch.from_numpy(init))
        info_d = _zeros((n_slots, 6))
        if levels is None:
            # launch plan: consecutive parts of the cost-ordered model list, each with its own kernel shape
            # (models per cluster x CTAs per cluster; 0x0 = first-generation kernel), each on its own
            # stream so that clusters of heavy models and dense packs of light models share the SMs
            parts = _cd_plan(C, n_slots, len(probs))
            tm_d = None
            if any(g for _, _, g, _ in parts):
                qh = np.array([p.Qc.data_ptr() for p in probs], dtype=np.uint64)
                tm_h = np.zeros(len(probs) * nat.lib().sglm_enet_cd_cluster_tmap_bytes(), dtype=np.uint8)
                rc_ = nat.lib().sglm_enet_cd_cluster_encode_tmaps(qh.ctypes.data_as(ctypes.c_void_p), len(probs), C,
                                                                  ldq, tm_h.ctypes.data_as(ctypes.c_void_p))
                if rc_ != 0:
                    raise nat.SglmNativeError("cd tensor maps: " + nat.lib().sglm_last_error().decode())
                tm_d = torch.from_numpy(tm_h).to("cuda")
            main = torch.cuda.current_stream()
            ready = torch.cuda.Event()
            ready.record(main)
            keep, side_done = [], []
            for pi, (r0, r1, gsz, csz) in enumerate(parts):
                if r1 <= r0:
                    continue
                st = main if pi == 0 else _side_stream(pi)
                if st is not main:
                    st.wait_event(ready)
                with torch.cuda.stream(st):
                    if gsz:
                        # groups of `gsz` models of the same problem (neighbours in the cost order, so that
                        # the members of a group run a similar number of sweeps), heaviest groups first
                        by_prob = {}
                        for r in range(r0, r1):
                            by_prob.setdefault(slot_prob[r], []).append(r)
                        groups = []
                        for p_, rows_ in by_prob.items():
                            for k in range(0, len(rows_), gsz):
                                chunk = rows_[k:k + gsz]
                                groups.append((chunk[0], p_, chunk + [-1] * (gsz - len(chunk))))
                        groups.sort(key=lambda g: g[0])
                        gp = _dev(np.array([g[1] for g in groups], dtype=np.int32), np.int32)
                        gs = _dev(np.array([g[2] for g in groups], dtype=np.int32).reshape(-1), np.int32)
                        gst = _zeros((len(groups), 2)) if CD_COLLECT_STATS else None
                        keep += [gp, gs]
                        if gst is not None:
                            cd_parts_log.append(dict(shape=(gsz, csz), slots=(r0, r1), group_stats=gst, info=info_d))
                        call("sglm_enet_cd_cluster_f64", ptr(Qp), ptr(qp), ptr(dp), ptr(yy), ldq, C, ptr(gp), ptr(gs),
                             ptr(pack_f[0]), ptr(pack_f[1]), ptr(pack_f[2]), ptr(pack_i[1]), len(groups), gsz, csz,
                             int(warm) | (int(CD_DEBUG_TIMER) << 8), int(do_screening), ptr(Wcd), ldw, ptr(info_d),
                             ptr(tm_d), ptr(gst), stream_ptr())
                    else:
                        if CD_COLLECT_STATS:
                            cd_parts_log.append(dict(shape=(0, 0), slots=(r0, r1), group_stats=None, info=info_d))
                        call("sglm_enet_cd_gram_f64", ptr(Qp), ptr(qp), ptr(dp), ptr(yy), ldq, C, ptr(pack_i[0][r0:]),
                             ptr(pack_f[0][r0:]), ptr(pack_f[1][r0:]), ptr(pack_f[2][r0:]), ptr(pack_i[1][r0:]),
                             r1 - r0, int(warm) | (int(CD_DEBUG_TIMER) << 8), int(do_screening), ptr(Wcd[r0:]), ldw,
                             ptr(info_d[r0:]), stream_ptr())
                    if st is not main:
                        ev = torch.cuda.Event()
                        ev.record(st)
                        side_done.append(ev)
            for ev in side_done:
                main.wait_event(ev)
        else:
            pred_t = _dev(pred, np.int64)
            for k, (a, b) in enumerate(levels):
                if k > 0:       # start every model of this path position from its predecessor's solution
                    Wcd[a:b] = Wcd.index_select(0, pred_t[a:b])
                call("sglm_enet_cd_gram_f64", ptr(Qp), ptr(qp), ptr(dp), ptr(yy), ldq, C, ptr(pack_i[0][a:]),
                     ptr(pack_f[0][a:]), ptr(pack_f[1][a:]), ptr(pack_f[2][a:]), ptr(pack_i[1][a:]), b - a,
                     int(k > 0), int(do_screening), ptr(Wcd[a:]), ldw, ptr(info_d[a:]), stream_ptr())
        real = [r for r, i in enumerate(slots) if i >= 0]
        dst = [slots[r] for r in real]
        W.index_copy_(0, _dev(dst, np.int64), Wcd.index_select(0, _dev(real, np.int64)))
        info[dst] = info_d.cpu().numpy()[real]
        status[dst] = (info[dst, 0] > info[dst, 1]).astype(np.int64)      # 1 = duality gap above tolerance
    groups = {}
    for i, m in enumerate(models):
        if m.kind in ("ridge", "ols"):
            groups.setdefault(id(m.problem), []).append(i)
    # one Cholesky launch per problem (one CTA per alpha): the launches of the problems of a grid are independent
    # and each fills only a few SMs, so they go to separate streams and run side by side.  Systems whose pivots
    # fell to rounding-noise level (rank-deficient least squares) or below zero are re-solved by the minimum-norm
    # solver on the same stream — decided on the device, no read-back (sglm_ols_minnorm_f64).
    launched = []
    if groups:
        main = torch.cuda.current_stream()
        mn_bytes = nat.lib().sglm_ols_minnorm_workspace_bytes(C)
    # first every buffer and host->device copy (on the main stream: a pageable copy blocks the host until the stream
    # reaches it, so none may be queued behind a wait on a side stream), then all launches
    prepared = []
    for gi, idxs in enumerate(groups.values()):
        p = models[idxs[0]].problem
        n_a = len(idxs)
        wb = nat.lib().sglm_ridge_workspace_bytes(C, p.ldq, n_a)
        alphas = _dev([0.0 if models[i].kind == "ols" else models[i].alpha for i in idxs], np.float64)
        work = torch.empty(wb // 8, dtype=torch.float64, device="cuda")
        Wr = _empty((n_a, ldw))
        st = torch.empty(n_a, dtype=torch.int32, device="cuda")
        has_ols = any(models[i].kind == "ols" for i in idxs)
        mn_work = torch.empty(mn_bytes // 8, dtype=torch.float64, device="cuda") if has_ols else None
        prepared.append((idxs, p, n_a, wb, alphas, work, Wr, st, mn_work))
    if groups:
        ready = torch.cuda.Event()
        ready.record(main)
    side_done = []
    for gi, (idxs, p, n_a, wb, alphas, work, Wr, st, mn_work) in enumerate(prepared):
        st_ = main if gi == 0 else _side_stream(100 + gi % 8)
        if st_ is not main:
            st_.wait_event(ready)
        with torch.cuda.stream(st_):
            call("sglm_ridge_solve_f64", ptr(p.Qc), p.ldq, ptr(p.qc), C, ptr(alphas), n_a, ptr(Wr), ldw, ptr(st),
                 ptr(work), wb, stream_ptr())
            for k, i in enumerate(idxs):
                # least squares (alpha == 0): rank deficiency is decided on the device — the launch returns at once
                # when every pivot was healthy.  (Ridge systems are positive definite; a failed one is re-solved
                # after the status read-back below, as scikit-learn falls back to its SVD solver.)
                if models[i].kind == "ols":
                    call("sglm_ols_minnorm_f64", ptr(p.Qc), p.ldq, ptr(p.qc), C, float(models[i].tol), 0.0, 3,
                         ctypes.c_void_p(st.data_ptr() + 4 * k), ptr(Wr[k]), ptr(mn_work), mn_bytes, stream_ptr())
            if st_ is not main:
                ev = torch.cuda.Event()
                ev.record(st_)
                side_done.append(ev)
                for t in (alphas, work, Wr, st, mn_work):
                    if t is not None:
                        t.record_stream(st_)
        launched.append((idxs, Wr, st, p, mn_work))
    for ev in side_done:
        main.wait_event(ev)
    for idxs, Wr, st, p, mn_work in launched:
        st_h = st.cpu().numpy()
        for k, i in enumerate(idxs):
            if (st_h[k] & 1) and models[i].kind == "ridge":
                # Cholesky met a non-positive pivot: the spectral solve, as sklearn's SVD fallback (_ridge.py:_solve_svd)
                if mn_work is None:
                    mn_work = torch.empty(mn_bytes // 8, dtype=torch.float64, device="cuda")
                call("sglm_ols_minnorm_f64", ptr(p.Qc), p.ldq, ptr(p.qc), C, 0.0, float(models[i].alpha), 1,
                     ctypes.c_void_p(st.data_ptr() + 4 * k), ptr(Wr[k]), ptr(mn_work), mn_bytes, stream_ptr())
        if np.any(st_h & 1):
            st_h = st.cpu().numpy()
        W.index_copy_(0, _dev(idxs, np.int64), Wr)
        # bit 1 alone (a tiny but positive pivot of a Ridge system) is not an error; bit 0 is cleared by the fallback
        status[idxs] = (st_h & 1) * 2                                 # 2 = not positive definite and not recovered
    del launched
    return W, info, status


def finalize(W, C, n_y, models):
    """Intercepts b = ybar - xbar.w and evaluation vectors V = [-w | e_y | -b]."""
    M = len(models)
    ldw = W.stride(0)
    ldv = _round_up(C + n_y + 1, 2)
    V = _empty((M, ldv))
    b = _empty((M,))
    ycol = _dev([m.problem.y_col for m in models], np.int32)
    xb = _dev(np.array([m.problem.xbar.data_ptr() for m in models], dtype=np.uint64).view(np.int64), np.int64)
    torch = nat.require_cuda()
    uniq, where = [], {}
    for m in models:
        if id(m.problem) not in where:
            where[id(m.problem)] = len(uniq)
            uniq.append(m.problem)
    ybar_p = torch.stack([p.scal for p in uniq])[:, 2].contiguous()
    yb = ybar_p.index_select(0, _dev([where[id(m.problem)] for m in models], np.int64)).contiguous()
    call("sglm_finalize_models_f64", ptr(W), ldw, C, n_y, ptr(ycol), ptr(xb), ptr(yb), M, ptr(b), ptr(V), ldv,
         stream_ptr())
    return b, V


QUADFORM_GEMM_MIN = 128     # vectors from which v'Av goes through the fp64 GEMM (below: the row-streaming kernel)


def quadform(A, V):
    """out[m] = V[m]' A V[m]."""
    M = V.shape[0]
    n = A.shape[0]
    if not M:
        return _empty((0,))
    if M >= QUADFORM_GEMM_MIN:
        # many vectors: one fp64 GEMM A V' (A streamed once per 64 vectors) + deterministic column dots
        torch = nat.require_cuda()
        ldb = _round_up(M, 64)
        Vt = _zeros((n, ldb))
        Vt[:, :M] = V[:, :n].t()
        Y = _empty((n, ldb))
        part = _empty((16, M))
        out = _empty((M,))
        call("sglm_quadform_gemm_f64", ptr(A), A.stride(0), n, ptr(Vt), ldb, M, ptr(Y), ptr(part), ptr(out), stream_ptr())
        return out
    # few models: split the rows of A over several CTAs per model group so that every SM streams a part
    groups = (M + 7) // 8
    splits = max(1, min(16, (2 * 148) // groups))
    if splits == 1:
        out = _empty((M,))
        call("sglm_quadform_f64", ptr(A), A.stride(0), n, ptr(V), V.stride(0), M, ptr(out), stream_ptr())
        return out
    part = _empty((splits, M))
    call("sglm_quadform_split_f64", ptr(A), A.stride(0), n, ptr(V), V.stride(0), M, splits, ptr(part), stream_ptr())
    return part.sum(dim=0)


# --------------------------------------------------------------------------- #
# explicit-matrix passes
# --------------------------------------------------------------------------- #
def _coef_dev(coef, intercept):
    w = _dev(np.asarray(coef, dtype=np.float64).reshape(-1), np.float64)
    b = _dev([float(np.asarray(intercept).reshape(-1)[0])], np.float64)
    return w, b


def predict(Xd, coef, intercept, link=0):
    T, C = Xd.shape
    w, b = _coef_dev(coef, intercept)
    if w.numel() != C:
        raise ValueError(f"X has {C} features, but the model was fitted with {w.numel()} features")
    out = _empty((T,))
    call("sglm_predict_f64", ptr(Xd), row_stride(Xd), T, C, ptr(w), ptr(b), link, ptr(out), stream_ptr())
    return out


def score_sums(Xd, yd, coef, intercept, link=0, rw=None, want_resid=False, power=None):
    """Fused pass: {n, sum r^2, sum y, sum y^2, sum y*eta, sum mu, sum y log y, sum r} (host).  With `power` (log link):
    the Tweedie family's deviance terms in slots 4..6 (sglm_score_glm_f64), the input of tweedie_d2_from_sums."""
    torch = nat.require_cuda()
    T, C = Xd.shape
    w, b = _coef_dev(coef, intercept)
    if w.numel() != C:
        raise ValueError(f"X has {C} features, but the model was fitted with {w.numel()} features")
    sums = _empty((8,))
    ws = torch.empty(nat.lib().sglm_score_workspace_bytes() // 8, dtype=torch.float64, device="cuda")
    resid = _empty((T,)) if want_resid else None
    if power is None:
        call("sglm_score_f64", ptr(Xd), row_stride(Xd), ptr(yd), ptr(rw), T, C, ptr(w), ptr(b), link, ptr(resid),
             ptr(sums), ptr(ws), stream_ptr())
    else:
        call("sglm_score_glm_f64", ptr(Xd), row_stride(Xd), ptr(yd), ptr(rw), T, C, ptr(w), ptr(b), float(power),
             ptr(resid), ptr(sums), ptr(ws), stream_ptr())
    return sums.cpu().numpy(), resid


def r2_from_sums(s):
    n, rss, sy, syy = s[0], s[1], s[2], s[3]
    tss = syy - sy * sy / n
    if tss <= 0.0:
        return 1.0 if rss == 0.0 else 0.0
    return float(1.0 - rss / tss)


def poisson_d2_from_sums(s):
    """D^2 = 1 - dev/dev_null (sklearn _glm/glm.py:387-463) from the fused sums."""
    n, sy, sy_eta, smu, sylogy = s[0], s[2], s[4], s[5], s[6]
    dev = 2.0 * (sylogy - sy_eta - sy + smu)
    ybar = sy / n
    dev_null = 2.0 * (sylogy - sy * np.log(ybar)) if ybar > 0 else 0.0
    return float(1.0 - dev / dev_null)


def tweedie_d2_from_sums(s, power):
    """D^2 = 1 - dev/dev_null of the Tweedie family of `power` (log link; TweedieRegressor.score,
    sklearn.metrics.d2_tweedie_score) from sums with the family's deviance terms {.., s4, s5, s6, ..}
    (sglm_score_glm_f64, sglm_glm_epilogue_f64 mode 1); the null model is mu = mean(y)."""
    if power == 1:
        return poisson_d2_from_sums(s)
    n, sy, s4, s5, s6 = s[0], s[2], s[4], s[5], s[6]
    ybar = sy / n
    if power == 2:
        dev = 2.0 * (s4 - s6 + s5 - n)
        dev_null = 2.0 * (n * np.log(ybar) - s6 + sy / ybar - n)
    else:
        p = float(power)
        c = s6 / ((1.0 - p) * (2.0 - p))
        dev = 2.0 * (c - s4 / (1.0 - p) + s5 / (2.0 - p))
        dev_null = 2.0 * (c - sy * ybar ** (1.0 - p) / (1.0 - p) + n * ybar ** (2.0 - p) / (2.0 - p))
    return float(1.0 - dev / dev_null)


# --------------------------------------------------------------------------- #
# (a9) Poisson by IRLS (Newton) — weighted statistics on the tensor path, Cholesky step
# --------------------------------------------------------------------------- #
POISSON_TC_PLANES = 4        # digit planes of the approximate Newton Hessian (4 x 7 bits)
POISSON_TC = None            # None: large problems; False: always the exact fp64 DMMA Gram (IRLS form)


def _poisson_tc(T, C):
    import os
    mode = os.environ.get("SGLM_POISSON_TC", "auto") if POISSON_TC is None else ("1" if POISSON_TC else "0")
    if mode in ("0", "1"):
        return mode == "1"
    return T * C * C >= (1 << 36)


def suffstats_tc_scaled(Xd, Yd, rs, max_planes, rows=None):
    """G = Z' diag(rs^2) Z, Z = [X | Y | 1], from at most `max_planes` digit planes per column (approximate when a
    column needs more): the weighted Gram of a Newton step on the tcgen05 path.  Returns G [1, n_aug, ldg]."""
    torch = nat.require_cuda()
    T, C = Xd.shape
    n_y = Yd.shape[1]
    n_aug = C + n_y + 1
    ldg = _round_up(n_aug, 8)
    colE = torch.empty(n_aug, dtype=torch.int32, device="cuda")
    colS = torch.empty(n_aug, dtype=torch.int32, device="cuda")
    scratch = torch.empty(n_aug, dtype=torch.int64, device="cuda")
    flag = torch.empty(1, dtype=torch.int32, device="cuda")
    call("sglm_gram_tc_analyze_scaled_f64", ptr(Xd), row_stride(Xd), ptr(Yd), row_stride(Yd), n_y, T, C, ptr(rs),
         int(max_planes), ptr(colE), ptr(colS), ptr(scratch), ptr(flag), stream_ptr())
    host = torch.cat([colS, flag]).cpu().numpy()
    if host[-1] != 0:
        raise ValueError("Input contains NaN, infinity or a value too large for dtype('float64').")
    colS_h = np.ascontiguousarray(host[:-1], dtype=np.int32)
    if rows is None:
        rows = torch.arange(T, dtype=torch.int64, device="cuda")
    pad = (-T) % 128
    if pad:
        rows = torch.cat([rows, torch.full((pad,), -1, dtype=torch.int64, device="cuda")])
    sizes = np.ascontiguousarray([T], dtype=np.int64)
    colS_p, sizes_p = colS_h.ctypes.data_as(ctypes.c_void_p), sizes.ctypes.data_as(ctypes.c_void_p)
    ws_bytes = nat.lib().sglm_gram_tc_workspace_bytes(n_aug, colS_p, 1, sizes_p)
    if ws_bytes == 0:
        raise nat.SglmNativeError("gram_tc: invalid plan")
    raw = torch.empty(ws_bytes + 1024, dtype=torch.uint8, device="cuda")
    off = (-raw.data_ptr()) % 1024
    G = _zeros((1, n_aug, ldg))
    call("sglm_gram_tc_scaled_f64", ptr(Xd), row_stride(Xd), ptr(Yd), row_stride(Yd), n_y, T, C, ptr(rs), ptr(colE),
         ptr(colS), colS_p, 1, sizes_p, ptr(rows), ptr(G), ldg, ctypes.c_void_p(raw.data_ptr() + off), ws_bytes,
         stream_ptr())
    return G


def suffstats_tc_scaled_sharded(Xd, Yd, rs, max_planes, all_reduce):
    """suffstats_tc_scaled when this process holds a SLICE of the rows (all_reduce as in suffstats_tc_sharded): the
    column analysis is combined over the processes (max / min), every process slices its rows and the int64 plane
    Grams are summed (exact), so G has the bits of the one-GPU weighted Gram over all rows, on every process."""
    torch = nat.require_cuda()
    T, C = Xd.shape
    n_y = Yd.shape[1]
    n_aug = C + n_y + 1
    ldg = _round_up(n_aug, 8)
    colmax = torch.empty(n_aug, dtype=torch.int64, device="cuda")
    colS = torch.empty(n_aug, dtype=torch.int32, device="cuda")
    colE = torch.empty(n_aug, dtype=torch.int32, device="cuda")
    flag = torch.empty(1, dtype=torch.int32, device="cuda")
    call("sglm_gram_tc_colstats_scaled_f64", ptr(Xd), row_stride(Xd), ptr(Yd), row_stride(Yd), n_y, T, C, ptr(rs),
         ptr(colmax), ptr(colS), stream_ptr())
    all_reduce(colmax, "max")
    all_reduce(colS, "min")
    call("sglm_gram_tc_exponents", ptr(colmax), n_aug, int(max_planes), ptr(colE), ptr(colS), ptr(flag), stream_ptr())
    host = torch.cat([colS, flag]).cpu().numpy()
    if host[-1] != 0:
        raise ValueError("Input contains NaN, infinity or a value too large for dtype('float64').")
    colS_h = np.ascontiguousarray(host[:-1], dtype=np.int32)
    rows = torch.full((max(_round_up(T, 128), 128),), -1, dtype=torch.int64, device="cuda")
    rows[:T] = torch.arange(T, dtype=torch.int64, device="cuda")
    sizes = np.ascontiguousarray([T], dtype=np.int64)
    member = np.ones((1, 1), dtype=np.int32)
    colS_p, sizes_p = colS_h.ctypes.data_as(ctypes.c_void_p), sizes.ctypes.data_as(ctypes.c_void_p)
    ws_bytes = nat.lib().sglm_gram_tc_cells_workspace_bytes(n_aug, colS_p, 1, sizes_p, 1)
    if ws_bytes == 0:
        raise nat.SglmNativeError("gram_tc: invalid plan")
    off_b, size_b = ctypes.c_uint64(0), ctypes.c_uint64(0)
    if nat.lib().sglm_gram_tc_cells_sgout(n_aug, colS_p, 1, sizes_p, 1, ctypes.byref(off_b), ctypes.byref(size_b)) != 0:
        raise nat.SglmNativeError("gram_tc: " + nat.lib().sglm_last_error().decode())
    raw = torch.empty(ws_bytes + 1024, dtype=torch.uint8, device="cuda")
    off = (-raw.data_ptr()) % 1024
    ws_p = ctypes.c_void_p(raw.data_ptr() + off)
    call("sglm_gram_tc_scaled_partial_f64", ptr(Xd), row_stride(Xd), ptr(Yd), row_stride(Yd), n_y, T, C, ptr(rs),
         ptr(colE), ptr(colS), colS_p, 1, sizes_p, ptr(rows), 1, member.ctypes.data_as(ctypes.c_void_p), ws_p, ws_bytes,
         stream_ptr())
    all_reduce(raw[off + off_b.value: off + off_b.value + size_b.value].view(torch.int64), "sum")
    G = _zeros((1, n_aug, ldg))
    call("sglm_gram_tc_cells_combine_f64", C, n_y, ptr(colE), ptr(colS), colS_p, 1, sizes_p, 1, ptr(G), ldg, ws_p, ws_bytes,
         stream_ptr())
    return G


def reduce_parts(parts, n_parts):
    """parts: n_parts equal contiguous blocks -> their element-wise sum, added in block order (sglm_reduce_parts_f64):
    the fixed-order sum of per-process partials gathered in process order."""
    n = parts.numel() // n_parts
    out = _empty((n,))
    call("sglm_reduce_parts_f64", ptr(parts), n, int(n_parts), ptr(out), stream_ptr())
    return out


def poisson_irls(Xd, yd, alpha, fit_intercept=True, rw=None, max_iter=100, tol=1e-4, coef_init=None,
                 intercept_init=None):
    """argmin mean(mu - y*eta) + alpha/2 |w|^2 (rows weighted by multiplicity rw).
    Newton/IRLS with step halving; stops after a Newton step below
    min(tol, 3e-6) * max(1, |w|_inf) (quadratic convergence: that iterate is ~1e-10 from the
    optimum) — i.e. at the optimum the reference's L-BFGS (gtol = tol) is heading for.  Returns (coef ndarray, intercept, n_iter)."""
    torch = nat.require_cuda()
    T, C = Xd.shape
    ldw = _round_up(C, 2)
    sums = _empty((8,))
    ws = torch.empty(nat.lib().sglm_score_workspace_bytes() // 8, dtype=torch.float64, device="cuda")
    weight = _empty((1, T))
    z = _empty((T, 1))
    if rw is None:
        n_tot, ysum = float(T), float(yd.sum().item())
    else:
        n_tot, ysum = float(rw.sum().item()), float((rw * yd).sum().item())
    if not (ysum > 0):
        raise ValueError("Some value(s) of y are out of the valid range of the loss 'HalfPoissonLoss'.")
    w = _zeros((ldw,))
    b = _zeros((1,))
    if coef_init is not None:
        w[:C] = _dev(np.asarray(coef_init, dtype=np.float64).reshape(-1), np.float64)
        if fit_intercept and intercept_init is not None:
            b[0] = float(intercept_init)
    elif fit_intercept:
        b[0] = float(np.log(ysum / n_tot))
    # Newton converges quadratically: once a step is below 3e-6 (relative), the iterate it produced is within
    # ~1e-10 of the optimum, so the confirming iteration (one more pass over X and one more weighted Gram, a
    # quarter of a warm-started fit) is not run.  The target stays "closer than 1e-8 to the optimum".
    step_tol = min(tol, 3e-6)
    w_prev, b_prev, f_prev = None, None, np.inf
    n_iter, halvings = 0, 0
    rows_hint = [n_tot]
    alphas = _dev([alpha * n_tot], np.float64)
    wb = nat.lib().sglm_ridge_workspace_bytes(C, _round_up(C, 8), 1)
    work = torch.empty(wb // 8, dtype=torch.float64, device="cuda")
    st = torch.empty(1, dtype=torch.int32, device="cuda")
    use_tc = _poisson_tc(T, C)
    refresh, last_step, hess, h11 = True, np.inf, None, None
    if use_tc:
        tc_rows = torch.arange(T, dtype=torch.int64, device="cuda")
        g_w = _empty((C,))
        xt_ws = torch.empty(nat.lib().sglm_xt_vec_workspace_bytes(C) // 8, dtype=torch.float64, device="cuda")
    while True:
        call("sglm_poisson_irls_prepare_f64", ptr(Xd), row_stride(Xd), ptr(yd), ptr(rw), T, C, ptr(w), ptr(b),
             ptr(weight), ptr(z), ptr(sums), ptr(ws), stream_ptr())
        f = float(sums[0].item()) / n_tot + 0.5 * alpha * float((w[:C] * w[:C]).sum().item())
        if w_prev is not None and not (f <= f_prev + 1e-12 * max(1.0, abs(f_prev))) and halvings < 30:
            w = 0.5 * (w + w_prev)
            b = 0.5 * (b + b_prev)
            halvings += 1
            refresh = True
            continue
        halvings = 0
        if n_iter >= max_iter:
            break
        if use_tc:
            # Newton step with an APPROXIMATE Hessian and the EXACT gradient: X'WX (with the weighted column sums
            # for the intercept) comes from the tcgen05 digit-plane Gram of sqrt(W) [X | z | 1] truncated to
            # POISSON_TC_PLANES planes (relative error 2^-28), the gradient X'(mu - y) from one fp64 pass over X.
            # (H~ + a n I) w_new = H~ w - g  has the same fixed point as the exact iteration (g + a n w = 0).
            # The factorised Hessian is kept while the steps keep shrinking fast (chord iterations: one pass
            # over X for the gradient and two triangular solves per step) and rebuilt when they do not.
            r = weight[0] - (yd if rw is None else rw * yd)                    # rw * (mu - y)
            call("sglm_xt_vec_f64", ptr(Xd), row_stride(Xd), ptr(r), T, C, ptr(g_w), ptr(xt_ws), xt_ws.numel() * 8,
                 stream_ptr())
            g_b = sums[1] - sums[3]
            w_new = _zeros((1, ldw))
            if refresh:
                rs = weight[0].sqrt()
                G = suffstats_tc_scaled(Xd, z, rs, POISSON_TC_PLANES, tc_rows)
                hess = center(G[0], None, C, 1, 0, fit_intercept)
                h11 = sums[1].clone()
                del G, rs
            rhs = hess.Qc[:, :C] @ w[:C] - g_w
            if fit_intercept:
                rhs = rhs + hess.xbar * g_b
            if refresh:
                hess.qc.copy_(rhs)
                call("sglm_ridge_solve_f64", ptr(hess.Qc), hess.ldq, ptr(hess.qc), C, ptr(alphas), 1, ptr(w_new), ldw,
                     ptr(st), ptr(work), wb, stream_ptr())
            else:
                call("sglm_chol_solve_f64", ptr(work), hess.ldq, C, 0, ptr(rhs.contiguous()), ptr(w_new), stream_ptr())
            b_new = _zeros((1,))
            if fit_intercept:
                b_new = b - g_b / h11 - (hess.xbar * (w_new[0, :C] - w[:C])).sum()
        else:
            G = suffstats(Xd, z, weight, rows_hint)
            p = center(G[0], None, C, 1, 0, fit_intercept)
            w_new = _zeros((1, ldw))
            call("sglm_ridge_solve_f64", ptr(p.Qc), p.ldq, ptr(p.qc), C, ptr(alphas), 1, ptr(w_new), ldw, ptr(st),
                 ptr(work), wb, stream_ptr())
            fetch_scalars([p])
            b_new = _zeros((1,))
            if fit_intercept:
                b_new[0] = p.ybar - float((p.xbar * w_new[0, :C]).sum().item())
        n_iter += 1
        dw = float((w_new[0, :C] - w[:C]).abs().max().item())
        db = float((b_new - b).abs().max().item())
        scale = max(1.0, float(w_new[0, :C].abs().max().item()))
        w_prev, b_prev, f_prev = w, b, f
        w, b = w_new[0].clone(), b_new
        step = max(dw, db) / scale
        if use_tc:
            # linear convergence (inexact Hessian): after a step s that contracted by rho = s / s_prev the iterate is
            # within s * rho / (1 - rho) of the optimum — stop when that bound is below min(tol, 1e-8)
            rho = min(step / last_step, 0.9) if np.isfinite(last_step) and last_step > 0 else 1.0
            if step * rho / (1.0 - min(rho, 0.9)) <= min(tol, 1e-8) or step <= 1e-12:
                break
        elif step <= step_tol:
            break
        refresh = step > 0.2 * last_step          # chord steps must keep contracting by 5x, else a new Hessian
        last_step = step
    return w[:C].cpu().numpy(), float(b.item()) if fit_intercept else 0.0, n_iter


# --------------------------------------------------------------------------- #
# (a9, batched) Poisson / Gamma / Tweedie grid: all (fold, alpha) fits advance together (csrc/poisson_batch.cu)
# --------------------------------------------------------------------------- #
PB_MAX_BATCH = 256       # models per batch (Eta is T x round_up(B, 64) doubles)
last_poisson_batch = None    # diagnostics of the most recent batch: iterations, Hessian refreshes, power, and for
                             # elastic-net models their number and the inner CD sweeps summed over models and rounds


class PoissonModel:
    """One fit of a batch: penalty alpha (r |w|_1 + (1 - r)/2 |w|^2) with r = l1_ratio (0: ridge), row-weight vector
    (index into RW, -1 = all rows), response column, and an optional start point (coef_init [C], intercept_init;
    default w = 0, b = log mean y)."""
    __slots__ = ("alpha", "fit_intercept", "rw", "ycol", "max_iter", "tol", "n_tot", "coef_init", "intercept_init",
                 "l1_ratio")

    def __init__(self, alpha, fit_intercept=True, rw=-1, ycol=0, max_iter=100, tol=1e-4, n_tot=None, coef_init=None,
                 intercept_init=None, l1_ratio=0.0):
        self.alpha, self.fit_intercept, self.rw, self.ycol = float(alpha), bool(fit_intercept), int(rw), int(ycol)
        self.max_iter, self.tol, self.n_tot = int(max_iter), float(tol), n_tot
        self.coef_init, self.intercept_init = coef_init, intercept_init
        self.l1_ratio = float(l1_ratio)


def _loss_name(power):
    return "HalfPoissonLoss" if power == 1 else "HalfTweedieLoss"


def _pb_hessian(Xd, y_col, rw_vec, w_ref, b_ref, fit_intercept, n_tot, use_tc, power=1.0, comm=None):
    """H~ = X' diag(rw v_ref) X (centred on the weighted column means when an intercept is fitted) with the Fisher
    weights v_ref = mu_ref^(2-p) of one reference model: the fused row pass gives the weights, the tcgen05 digit-plane
    Gram (large problems) or the fp64 DMMA Gram the matrix.  Returns (Problem-like hess with Qc / xbar, h11 = sum of
    the weights as a device scalar).  With `comm` (rows sharded over processes, see tweedie_grid_batched) the Gram
    is the staged one summed over the processes (tcgen05) or the combined fp64 partials, h11 the combined sum."""
    torch = nat.require_cuda()
    T, C = Xd.shape
    sums = _empty((8,))
    ws = torch.empty(nat.lib().sglm_score_workspace_bytes() // 8, dtype=torch.float64, device="cuda")
    weight = _empty((1, T))
    z = _empty((T, 1))
    call("sglm_glm_irls_prepare_f64", ptr(Xd), row_stride(Xd), ptr(y_col), ptr(rw_vec), T, C, ptr(w_ref), ptr(b_ref),
         float(power), ptr(weight), ptr(z), ptr(sums), ptr(ws), stream_ptr())
    if comm is not None:
        if use_tc:
            G = suffstats_tc_scaled_sharded(Xd, z, weight[0].sqrt(), POISSON_TC_PLANES, comm.all_reduce)
        else:
            G = comm.combine(suffstats(Xd, z, weight, [n_tot]))
        return center(G[0], None, C, 1, 0, fit_intercept), comm.combine(sums[1:2])
    if use_tc:
        G = suffstats_tc_scaled(Xd, z, weight[0].sqrt(), POISSON_TC_PLANES)
    else:
        G = suffstats(Xd, z, weight, [n_tot])
    hess = center(G[0], None, C, 1, 0, fit_intercept)
    return hess, sums[1:2].clone()


def poisson_grid_batched(Xd, Yd, models, RW=None):
    """Fit every PoissonModel of `models` on (Xd, Yd[:, ycol]) with row weights RW[rw] — argmin mean(mu - y eta) +
    alpha/2 |w|^2 over the weighted rows — as ONE batched iteration (see csrc/poisson_batch.cu).  Returns
    (W [B, C] CUDA, b [B] CUDA, n_iter [B] host, status [B] host: 1 converged, 2 max_iter)."""
    return tweedie_grid_batched(Xd, Yd, models, RW, 1.0)


def tweedie_grid_batched(Xd, Yd, models, RW=None, power=1.0, comm=None):
    """poisson_grid_batched for the Tweedie family of `power` (1, or > 1; log link): argmin mean(l(y, eta)) +
    alpha/2 |w|^2 with sklearn's HalfTweedieLoss l (p = 2: Gamma, whose Fisher Hessian X' diag(rw) X does not depend
    on the iterate and is built once per fold).  A model with l1_ratio r > 0 has the elastic-net penalty
    alpha r |w|_1 + alpha (1 - r)/2 |w|^2 and takes proximal-Newton steps (sglm_pb_step_enet_f64); it may share a
    batch with ridge models, whose steps are unchanged.

    comm: the rows are sharded over processes — Xd, Yd and RW hold this process's rows, every process calls with the
    same models — and `comm` combines the cross-row reductions: all_reduce(t, op) in place for the integer
    collectives of the tcgen05 Gram (op "max" / "min" / "sum"; also "min" on fp64), combine(t) = the fp64 partials
    of all processes added in process order (every process gets the same bits).  Every process then holds every
    model's coefficients; all host decisions are taken on combined values, so the processes stay in lock step."""
    torch = nat.require_cuda()
    global last_poisson_batch
    power = float(power)
    if not (power == 1.0 or power > 1.0):
        raise NotImplementedError(f"power={power}: the batched GLM solver covers power 1 and power > 1 (log link)")
    T, C = Xd.shape
    out_W, out_b, out_it, out_st = [], [], [], []
    diag = []
    for c0 in range(0, len(models), PB_MAX_BATCH):
        Wb, bb, it, st, dg = _poisson_batch(Xd, Yd, models[c0:c0 + PB_MAX_BATCH], RW, power, comm)
        out_W.append(Wb); out_b.append(bb); out_it.append(it); out_st.append(st); diag.append(dg)
    last_poisson_batch = diag
    return torch.cat(out_W), torch.cat(out_b), np.concatenate(out_it), np.concatenate(out_st)


def _poisson_batch(Xd, Yd, models, RW, power, comm=None):
    torch = nat.require_cuda()
    T, C = Xd.shape
    B = len(models)
    ldb = _round_up(B, 64)
    ldw = _round_up(C, 2)
    ldy = Yd.stride(0)
    n_w = 0 if RW is None else RW.shape[0]
    # ---- per-model constants: rows in the fit, weighted mean of y (start point b = log ybar, sklearn glm.py:264-270)
    ycontig = {}
    combos = sorted({(m.rw, m.ycol) for m in models})
    stats = torch.stack([torch.stack([(RW[rw].sum() if rw >= 0 else torch.tensor(float(T), device="cuda", dtype=torch.float64)),
                                      ((RW[rw] * Yd[:, yc]).sum() if rw >= 0 else Yd[:, yc].sum()),
                                      Yd[:, yc].min() if T else torch.tensor(np.inf, device="cuda", dtype=torch.float64)])
                         for rw, yc in combos])
    T_all = T
    if comm is not None:
        # counts and sums of y over all processes (+ the total row count, which picks the Hessian path), min y
        sums_ = comm.combine(torch.cat([stats[:, :2].reshape(-1), torch.tensor([float(T)], device="cuda", dtype=torch.float64)]))
        T_all = int(sums_[-1].item())
        ymin = stats[:, 2].contiguous()
        comm.all_reduce(ymin, "min")
        stats = torch.cat([sums_[:-1].reshape(-1, 2), ymin[:, None]], dim=1)
    stats = stats.cpu().numpy()
    info = {k: v for k, v in zip(combos, stats)}
    if any(v[2] < 0 for v in info.values()) or any(not (v[1] > 0) for v in info.values()) or \
            (power >= 2 and any(not (v[2] > 0) for v in info.values())):
        raise ValueError(f"Some value(s) of y are out of the valid range of the loss '{_loss_name(power)}'.")
    n_tot = np.array([info[(m.rw, m.ycol)][0] for m in models])
    b0 = np.array([np.log(info[(m.rw, m.ycol)][1] / info[(m.rw, m.ycol)][0]) if m.fit_intercept else 0.0 for m in models])
    for yc in {m.ycol for m in models}:
        ycontig[yc] = Yd[:, yc].contiguous()
    # ---- state on the device
    f64, i32 = np.float64, np.int32
    warm = [i for i, m in enumerate(models) if m.coef_init is not None]
    for i in warm:
        if models[i].fit_intercept and models[i].intercept_init is not None:
            b0[i] = float(np.asarray(models[i].intercept_init, dtype=f64).reshape(-1)[0])
    W, Wprev, Wnew, rhs = (_zeros((B, ldw)) for _ in range(4))
    for i in warm:
        W[i, :C] = _dev(np.asarray(models[i].coef_init, dtype=f64).reshape(-1), f64)
    b = _dev(b0, f64)
    bprev, fprev, fcur, last_step, step_out = (_zeros((B,)) for _ in range(5))
    ratio_out = torch.ones(B, dtype=torch.float64, device="cuda")        # 1.0 = contraction not known yet
    zi = lambda: torch.zeros(B, dtype=torch.int32, device="cuda")
    halv, n_iter, status, flag, has_prev = zi(), zi(), zi(), zi(), zi()
    alpha = _dev([m.alpha for m in models], f64)
    l1r = _dev([m.l1_ratio for m in models], f64)
    n_tot_d = _dev(n_tot, f64)
    tol = _dev([m.tol for m in models], f64)
    fit_icpt = _dev([int(m.fit_intercept) for m in models], i32)
    max_iter = _dev([m.max_iter for m in models], i32)
    groups = {}
    for i, m in enumerate(models):
        groups.setdefault((m.rw, m.fit_intercept), []).append(i)
    gkeys = list(groups)
    hess_id = _dev([gkeys.index((m.rw, m.fit_intercept)) for m in models], i32)
    ycol = _dev([m.ycol for m in models], i32)
    rw_a = _dev([m.rw for m in models], i32)
    red = _zeros((C * ldb + B * 4,))        # the cross-row reductions of an iteration, combined in one call under comm
    Gw = red[:C * ldb].view(C, ldb)
    sums = red[C * ldb:].view(B, 4)
    Wt = _zeros((C, ldb))
    Eta = _empty((max(T, 1), ldb))
    xt_bytes = nat.lib().sglm_pb_gemm_tn_workspace_bytes(T, C, ldb)
    xt_ws = torch.empty(xt_bytes // 8 + 1, dtype=torch.float64, device="cuda")
    ep_bytes = nat.lib().sglm_pb_epilogue_workspace_bytes(T, B)
    ep_ws = torch.empty(ep_bytes // 8 + 1, dtype=torch.float64, device="cuda")
    ldq = _round_up(C, 8)
    # ---- Hessians (one per fold / intercept setting) and the factors of (H~ + alpha n I) of every model
    use_tc = _poisson_tc(T_all, C)
    n_h = len(gkeys)
    HQ = torch.zeros(n_h, dtype=torch.int64, device="cuda")
    Hxbar = torch.zeros(n_h, dtype=torch.int64, device="cuda")
    Hh11 = _zeros((n_h,))
    L_of = torch.zeros(B, dtype=torch.int64, device="cuda")
    keep = {}
    wb_of = {}

    refreshed_at = {g: 0 for g in range(n_h)}
    n_refresh = {g: 1 for g in range(n_h)}

    def refresh(g, ref):
        """New H~ of group g from the current iterate of model `ref`, new factors for the group's models."""
        rw, fi = gkeys[g]
        idxs = groups[gkeys[g]]
        rw_vec = RW[rw] if rw >= 0 else None
        hess, h11 = _pb_hessian(Xd, ycontig[models[ref].ycol], rw_vec, W[ref], b[ref:ref + 1], fi, float(n_tot[ref]), use_tc,
                                power, comm)
        an = _dev([models[i].alpha * n_tot[i] if models[i].l1_ratio == 0 else
                   models[i].alpha * (1.0 - models[i].l1_ratio) * n_tot[i] for i in idxs], f64)
        wb = nat.lib().sglm_ridge_workspace_bytes(C, hess.ldq, len(idxs))
        work = torch.empty(wb // 8, dtype=torch.float64, device="cuda")
        Wtmp = _empty((len(idxs), ldw))
        st = torch.empty(len(idxs), dtype=torch.int32, device="cuda")
        call("sglm_ridge_solve_f64", ptr(hess.Qc), hess.ldq, ptr(hess.qc), C, ptr(an), len(idxs), ptr(Wtmp), ldw, ptr(st),
             ptr(work), wb, stream_ptr())
        keep[g] = (hess, work, h11)           # the previous Hessian / factors of the group are released here
        HQ[g] = hess.Qc.data_ptr()
        Hxbar[g] = hess.xbar.data_ptr()
        Hh11[g:g + 1] = h11
        stride = (C + 1) * hess.ldq * 8
        L_of[_dev(idxs, np.int64)] = _dev([work.data_ptr() + k * stride for k in range(len(idxs))], np.int64)
        sel = _dev(idxs, np.int64)
        last_step[sel] = 0.0                      # the contraction estimate restarts with the new Hessian
        ratio_out[sel] = 1.0
        if g in borrowed:                         # the group now has its own Hessian
            hess_id[sel] = hess_true[sel]
            hscale[sel] = 1.0
            del borrowed[g]

    # First step: every model starts from w = 0, b = log(mean y), where the Hessian is mean(y)^(2-p) * X'X over the
    # model's rows.  A fold whose parameter sets also have a full-data model (the refit of every CV set) borrows that
    # group's Hessian and factors for this one step, scaled by n_f mean_f(y)^(2-p) / (n mean(y)^(2-p)) (p = 1: its
    # share of sum(y)) — 1 weighted Gram and 1 factorisation per alpha instead of one per (fold, alpha); its own
    # Hessian follows with the refresh after the first step.  Warm-started models start elsewhere and borrow nothing.
    hscale = torch.ones(B, dtype=torch.float64, device="cuda")
    borrowed = {}
    for g, (rw, fi) in enumerate(gkeys):
        if rw < 0 or (-1, fi) not in groups:
            continue
        g0 = gkeys.index((-1, fi))
        by_alpha = {(models[i].alpha, models[i].l1_ratio, models[i].ycol == 0): i for i in groups[gkeys[g0]]}
        pairs = [(i, by_alpha.get((models[i].alpha, models[i].l1_ratio, True))) for i in groups[gkeys[g]]]
        if all(j is not None and models[i].coef_init is None and models[j].coef_init is None for i, j in pairs):
            borrowed[g] = (g0, pairs)
    for g in range(n_h):
        if g not in borrowed:
            refresh(g, groups[gkeys[g]][0])
    hess_true = hess_id.clone()
    for g, (g0, pairs) in borrowed.items():
        mine = _dev([i for i, _ in pairs], np.int64)
        theirs = _dev([j for _, j in pairs], np.int64)
        hess_id[mine] = g0
        L_of[mine] = L_of[theirs]
        if power == 1:
            share = np.array([info[(models[i].rw, models[i].ycol)][1] / info[(models[j].rw, models[j].ycol)][1] for i, j in pairs])
        else:
            def scale(k):
                n_k, sy_k = info[(models[k].rw, models[k].ycol)][:2]
                return n_k * (sy_k / n_k) ** (2.0 - power)
            share = np.array([scale(i) / scale(j) for i, j in pairs])
        hscale[mine] = _dev(share, f64)
    n_words = nat.lib().sglm_pb_state_words()
    fields = [W, Wprev, Wnew, rhs, b, bprev, fprev, fcur, last_step, step_out, ratio_out, halv, n_iter, status, flag,
              has_prev, alpha, n_tot_d, tol, fit_icpt, max_iter, hess_id, HQ, Hxbar, Hh11, sums, Gw, hscale]
    words = [t.data_ptr() for t in fields] + [ldw, ldq, ldb, C | (B << 32)]
    if len(words) != n_words:
        raise nat.SglmNativeError(f"poisson batch: state layout mismatch ({len(words)} words, library expects {n_words})")
    state = np.array(words, dtype=np.uint64)
    state_p = state.ctypes.data_as(ctypes.c_void_p)
    RWp, ldrw = (ptr(RW), RW.stride(0)) if RW is not None else (None, 0)
    enet = [i for i, m in enumerate(models) if m.l1_ratio != 0]
    if enet:
        enet_idx = _dev(enet, i32)
        en_bytes = nat.lib().sglm_pb_enet_workspace_bytes(C, ldw, len(enet))
        en_ws = torch.empty(en_bytes // 8 + 1, dtype=torch.float64, device="cuda")
        en_info = _zeros((len(enet), 6))
        sweeps = torch.zeros((), dtype=torch.float64, device="cuda")
    it = 0
    max_rounds = int(max(m.max_iter for m in models)) + 40
    while it < max_rounds:
        Wt[:, :B] = W[:, :C].t()
        call("sglm_pb_eta_f64", ptr(Xd), row_stride(Xd), T, C, ptr(Wt), ldb, ptr(Eta), stream_ptr())
        call("sglm_glm_epilogue_f64", ptr(Eta), ldb, B, T, ptr(Yd), ldy, ptr(ycol), RWp, ldrw, ptr(rw_a), None, ptr(b),
             ptr(status), power, 0, ptr(sums), ptr(ep_ws), ep_ws.numel() * 8, stream_ptr())
        call("sglm_pb_xt_r_f64", ptr(Xd), row_stride(Xd), T, C, ptr(Eta), ldb, ptr(Gw), ptr(xt_ws), xt_ws.numel() * 8,
             stream_ptr())
        if comm is not None:
            red.copy_(comm.combine(red))
        if enet:
            call("sglm_pb_step_enet_f64", state_p, ptr(L_of), ptr(l1r), ptr(enet_idx), len(enet), ptr(en_ws), en_ws.numel() * 8,
                 ptr(en_info), stream_ptr())
            sweeps += en_info[:, 2].sum()
        else:
            call("sglm_pb_step_f64", state_p, ptr(L_of), stream_ptr())
        it += 1
        host = torch.stack([status.to(torch.float64), step_out, ratio_out]).cpu().numpy()     # the one read-back per iteration
        st_h, step_h, ratio_h = host[0], host[1], host[2]
        if np.all(st_h != 0):
            break
        # refresh policy: after the first step (the start Hessian belongs to mu = const), then whenever the steps of a
        # fold stop contracting by at least 3x per iteration; reference = the active model with the largest step.
        # Gamma (Fisher weight 1): a group's own Hessian is exact for every iterate, only a borrowed one is replaced.
        for g in range(n_h):
            if power == 2 and g not in borrowed:
                continue
            idxs = np.array(groups[gkeys[g]])
            act = idxs[st_h[idxs] == 0]
            if len(act) == 0 or n_refresh[g] >= 8:
                continue
            taken = act[step_h[act] > 0]
            slow = len(taken) and np.max(ratio_h[taken]) > 0.35 and np.max(step_h[taken]) > 1e-7
            if (n_refresh[g] == 1 and it >= 1) or (slow and it - refreshed_at[g] >= 2):
                ref = int(act[np.argmax(np.abs(step_h[act]))])
                refresh(g, ref)
                refreshed_at[g], n_refresh[g] = it, n_refresh[g] + 1
    n_it = n_iter.cpu().numpy().astype(np.int64)
    st_f = status.cpu().numpy().astype(np.int64)
    st_f[st_f == 0] = 2
    diag = dict(rounds=it, refreshes=dict(n_refresh), models=B, hessian_groups=n_h, tensor_core_hessian=bool(use_tc),
                power=power)
    if enet:
        diag.update(enet_models=len(enet), inner_sweeps=int(sweeps.item()))
    return W[:, :C].contiguous(), b.clone(), n_it, st_f, diag


def poisson_scores_batched(Xd, Yd, W, b, ycol, rw_a, rw_b, RW):
    """Score sums of B fitted Poisson models in one pass over X: sums [B, 2, 8] (host) for the row weights rw_a /
    rw_b of each model (-1: all rows; rw_b = -2: none) — {n, sum r^2, sum y, sum y^2, sum y eta, sum mu,
    sum y log y, sum r}, the inputs of D^2 / -MSE / pooled R^2 (sglm_score_f64 semantics)."""
    return tweedie_scores_batched(Xd, Yd, W, b, ycol, rw_a, rw_b, RW, 1.0)


def tweedie_scores_batched(Xd, Yd, W, b, ycol, rw_a, rw_b, RW, power, comm=None):
    """poisson_scores_batched for the Tweedie family of `power`: slots 4..6 hold the family's deviance terms
    (sglm_score_glm_f64 semantics), the input of tweedie_d2_from_sums.  comm: rows sharded over processes, the sums
    combined (tweedie_grid_batched)."""
    torch = nat.require_cuda()
    T, C = Xd.shape
    B = W.shape[0]
    out = np.zeros((B, 2, 8))
    for c0 in range(0, B, PB_MAX_BATCH):
        n = min(PB_MAX_BATCH, B - c0)
        ldb = _round_up(n, 64)
        Wt = _zeros((C, ldb))
        Wt[:, :n] = W[c0:c0 + n, :C].t()
        Eta = _empty((max(T, 1), ldb))
        call("sglm_pb_eta_f64", ptr(Xd), row_stride(Xd), T, C, ptr(Wt), ldb, ptr(Eta), stream_ptr())
        sums = _zeros((n, 16))
        ep_bytes = nat.lib().sglm_pb_epilogue_workspace_bytes(T, n)
        ep_ws = torch.empty(ep_bytes // 8 + 1, dtype=torch.float64, device="cuda")
        # named tensors: a temporary freed inside the argument list would hand its block to the next allocation
        ids = _dev(np.stack([ycol[c0:c0 + n], rw_a[c0:c0 + n], rw_b[c0:c0 + n]]), np.int32)
        b_part = b[c0:c0 + n].contiguous()
        call("sglm_glm_epilogue_f64", ptr(Eta), ldb, n, T, ptr(Yd), Yd.stride(0), ptr(ids[0]),
             ptr(RW) if RW is not None else None, RW.stride(0) if RW is not None else 0,
             ptr(ids[1]), ptr(ids[2]), ptr(b_part), None, float(power), 1, ptr(sums), ptr(ep_ws), ep_ws.numel() * 8,
             stream_ptr())
        if comm is not None:
            sums = comm.combine(sums)
        out[c0:c0 + n] = sums.cpu().numpy().reshape(n, 2, 8)
    return out
