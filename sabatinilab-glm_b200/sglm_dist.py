"""
sglm_dist — multi-GPU sharding of the CV grid (one process per GPU, torch.distributed).

The reference has no distributed backend (single process, Python threads).  The grid shards
naturally: every parameter set — its F fold fits plus the full-data refit — is independent
of every other (backend/sglm_cv.py:131, :308 already treats them as separate queue items).
So parameter sets are dealt round-robin (in cost order) to the ranks, every rank builds
the statistics of the shared design locally, and the only collectives are

    broadcast  : the inputs from rank `src` (base signals / design, response, fold indices)
    all_gather : the per-set result records (coefficients, intercepts, scores)

— no collective inside the data path.  NCCL carries the tensors when the process group is
NCCL (NVLink 5 / NVSwitch on a B200 box); the same code runs over gloo on CPU tensors,
which is how tests/test_dist_gloo.py exercises it with world_size = 2.

`compute` is the per-rank engine: by default the B200 batched plan of sglm_cv; tests inject
the CPU oracle so that the sharding / ordering / selection logic is checked without a GPU.
"""
import numpy as np


def _dist():
    import torch.distributed as dist
    return dist


def shard_indices(n_items, world_size, rank, cost=None):
    """Indices of the items owned by `rank`: items sorted by decreasing cost and dealt
    round-robin, so every rank gets a similar mix of expensive (weakly regularised) and
    cheap parameter sets."""
    order = np.arange(n_items) if cost is None else np.argsort(-np.asarray(cost, dtype=np.float64), kind="stable")
    return sorted(int(i) for i in order[rank::world_size])


def default_cost(glm_kwargs):
    """Heuristic work estimate of one parameter set: coordinate descent on a weak penalty
    needs many sweeps; direct solvers (alpha == 0 or l1_ratio == 0) are cheap."""
    a = float(glm_kwargs.get("alpha", 1.0))
    l1 = float(glm_kwargs.get("l1_ratio", 0.5))
    if a == 0.0 or l1 == 0.0:
        return 0.0
    return 1.0 / max(a * max(l1, 1e-3), 1e-12)


def broadcast_inputs(X, y, cv_idx, src=0, group=None, device=None):
    """Broadcast (X, y, cv_idx) from rank `src`.  Non-source ranks pass None.  Tensors travel
    over the group's backend (NCCL: device tensors; gloo: CPU tensors)."""
    import torch
    dist = _dist()
    rank = dist.get_rank(group)
    meta = [None]
    if rank == src:
        Xt = torch.as_tensor(X, dtype=torch.float64)
        yt = torch.as_tensor(y, dtype=torch.float64).reshape(-1)
        meta = [dict(x_shape=tuple(Xt.shape), n_y=int(yt.numel()),
                     folds=[(int(len(a)), int(len(b))) for a, b in cv_idx])]
    dist.broadcast_object_list(meta, src=src, group=group)
    m = meta[0]
    dev = device if device is not None else ("cuda" if dist.get_backend(group) == "nccl" else "cpu")
    if rank == src:
        Xt, yt = Xt.to(dev).contiguous(), yt.to(dev).contiguous()
        idx = [(torch.as_tensor(np.asarray(a), dtype=torch.int64).to(dev),
                torch.as_tensor(np.asarray(b), dtype=torch.int64).to(dev)) for a, b in cv_idx]
    else:
        Xt = torch.empty(m["x_shape"], dtype=torch.float64, device=dev)
        yt = torch.empty(m["n_y"], dtype=torch.float64, device=dev)
        idx = [(torch.empty(na, dtype=torch.int64, device=dev), torch.empty(nb, dtype=torch.int64, device=dev))
               for na, nb in m["folds"]]
    dist.broadcast(Xt, src=src, group=group)
    dist.broadcast(yt, src=src, group=group)
    for a, b in idx:
        dist.broadcast(a, src=src, group=group)
        dist.broadcast(b, src=src, group=group)
    return Xt, yt, idx


def _b200_compute(X, y, cv_idx, entries, score_method):
    import sglm_cv
    return sglm_cv._cv_batch(X, y, cv_idx, entries, None, None, score_method)


def _record(r):
    """Picklable, device-free record of one result dict (the fitted model travels as its
    coefficients; it is rebuilt on the receiving side)."""
    m = r["model"]
    return {k: r[k] for k in ("cv_coefs", "cv_intercepts", "cv_scores_train", "cv_scores_test",
                              "cv_mean_score_train", "cv_mean_score", "cv_std_score", "cv_R2_score",
                              "cv_mse_score", "glm_kwargs")} | {
        "coef_": np.asarray(m.coef_), "intercept_": float(np.asarray(m.intercept_).reshape(-1)[0])}


def cv_glm_mult_params_sharded(X, y, cv_idx, model_name, glm_kwarg_lst, verbose=0, score_method='mse',
                               group=None, compute=None, rebuild_model=None):
    """Distributed `cv_glm_mult_params`: every rank calls it with the same arguments (use
    `broadcast_inputs` first when only one rank holds the data).  Returns, on every rank, the
    reference's result dict (backend/sglm_cv.py:420-426) with `full_cv_results` in the order
    of `glm_kwarg_lst` and the reference's strict-'>' selection."""
    dist = _dist()
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    compute = compute or _b200_compute
    entries = []
    for kw in glm_kwarg_lst:
        name = kw.pop('model_name', 'Gaussian')                    # backend/sglm_cv.py:288
        entries.append((name, kw))
    mine = shard_indices(len(entries), world, rank, [default_cost(kw) for _, kw in entries])
    local = compute(X, y, cv_idx, [entries[i] for i in mine], score_method) if mine else []
    payload = [(i, _record(r)) for i, r in zip(mine, local)]
    gathered = [None] * world
    dist.all_gather_object(gathered, payload, group=group)
    records = [None] * len(entries)
    for part in gathered:
        for i, rec in part:
            records[i] = rec
    for (name, kw), rec in zip(entries, records):                  # 'roll' was popped on the owning rank only
        kw.pop('roll', None)
        rec["glm_kwargs"] = kw
    resp = []
    for (name, kw), rec in zip(entries, records):
        out = dict(rec)
        coef, icpt = out.pop("coef_"), out.pop("intercept_")
        out["model"] = rebuild_model(name, kw, coef, icpt) if rebuild_model else _rebuild(name, kw, coef, icpt)
        resp.append(out)
    best_score, best = -np.inf, None
    for r in resp:
        s = r['cv_R2_score'] if score_method == 'r2' else r['cv_mean_score']
        if score_method in ('r2', 'mse') and s > best_score:
            best_score, best = s, r
    return {'best_score': best_score, 'best_score_std': best['cv_std_score'], 'best_params': best['glm_kwargs'],
            'best_model': best['model'], 'full_cv_results': resp}


def _rebuild(model_name, kw, coef, intercept):
    import sglm_
    glm = sglm_.GLM(model_name, **kw)
    glm.model.coef_ = np.asarray(coef, dtype=np.float64)
    glm.model.intercept_ = float(intercept)
    glm.coef_ = glm.beta_ = glm.model.coef_
    glm.intercept_ = glm.beta0_ = glm.model.intercept_
    return glm


# --------------------------------------------------------------------------- #
# ONE grid strong-scaled over the GPUs of a box (north star: "a full CV grid ... completes on 8 x B200")
# --------------------------------------------------------------------------- #
last_timeline = None       # {stage: ms} of the most recent cv_grid_strong call on this rank (CUDA events)


def deal_models(costs, world_size):
    """Owner rank of every model: models sorted by decreasing cost and dealt in a snake (0..N-1, N-1..0, ...), so
    every rank gets the same number of models (+-1) and a similar mix of heavy and light ones.  Returns
    (owner[M], order[M]) with order = model indices from the most to the least expensive."""
    costs = np.asarray(costs, dtype=np.float64)
    order = np.argsort(-costs, kind="stable")
    owner = np.empty(len(costs), dtype=np.int64)
    for j, i in enumerate(order):
        lap, pos = divmod(j, world_size)
        owner[i] = pos if lap % 2 == 0 else world_size - 1 - pos
    return owner, order


def model_cost(spec):
    """Work estimate of one fit: weakly penalised coordinate descent is heavy-tailed, direct solves are cheap."""
    if spec.kind in ("ridge", "ols"):
        return 0.0
    return 1.0 / max(spec.alpha * max(spec.l1_ratio, 1e-3), 1e-300)


def pack_results(W, b, rss_full, rss_test, rss_train, info, status, n_pad):
    """One [n_pad, C + 10] tensor per rank: [coef (C) | intercept | rss_full | rss_test | rss_train | info (6) |
    status]; `info` / `status` are host arrays, the rest tensors on W's device."""
    import torch
    n, C = W.shape
    out = torch.zeros((n_pad, C + 11), dtype=torch.float64, device=W.device)
    if n:
        out[:n, :C] = W
        out[:n, C] = b
        out[:n, C + 1] = rss_full
        out[:n, C + 2] = rss_test
        out[:n, C + 3] = rss_train
        out[:n, C + 4:C + 10] = torch.from_numpy(np.ascontiguousarray(info, dtype=np.float64)).to(W.device)
        out[:n, C + 10] = torch.from_numpy(np.ascontiguousarray(status, dtype=np.float64)).to(W.device)
    return out


def unpack_results(gathered, owner_lists, C):
    """gathered [world, n_pad, C + 11] + the model indices each rank owned (in its local order) -> per-model
    arrays in global model order."""
    import torch
    M = sum(len(o) for o in owner_lists)
    index = torch.empty(M, dtype=torch.int64)
    pos = 0
    n_pad = gathered.shape[1]
    for r, mine in enumerate(owner_lists):
        index[pos:pos + len(mine)] = r * n_pad + torch.arange(len(mine))
        pos += len(mine)
    flat = gathered.reshape(-1, C + 11).index_select(0, index.to(gathered.device))
    dest = torch.from_numpy(np.concatenate([np.asarray(o, dtype=np.int64) for o in owner_lists]) if M else np.zeros(0, np.int64))
    full = torch.empty_like(flat)
    full.index_copy_(0, dest.to(flat.device), flat)
    return full


class RankComm:
    """The cross-row reductions of a row-sharded computation over the ranks of `group` (NCCL, device tensors):
    all_reduce(t, op) in place (op "max" / "min" / "sum"), and combine(t) = the fp64 tensors of all ranks gathered and
    added in rank order on the device (_engine.reduce_parts) — every rank gets the same bits, which an fp64 all-reduce
    does not promise."""

    def __init__(self, group=None):
        dist = _dist()
        self.group = group
        self.world = dist.get_world_size(group)

    def all_reduce(self, t, op):
        dist = _dist()
        dist.all_reduce(t, op={"max": dist.ReduceOp.MAX, "min": dist.ReduceOp.MIN, "sum": dist.ReduceOp.SUM}[op],
                        group=self.group)

    def combine(self, t):
        import torch
        import _engine as eng
        flat = t.reshape(-1).contiguous()
        parts = torch.empty(self.world * flat.numel(), dtype=flat.dtype, device=flat.device)
        _dist().all_gather_into_tensor(parts, flat, group=self.group)
        return eng.reduce_parts(parts, self.world).reshape(t.shape)


LOG_LINK_KINDS = ("poisson", "tweedie", "tweedie_enet")
GAUSSIAN_KINDS = ("ols", "ridge", "lasso", "enet")


def cv_grid_strong(X0, shift_amt_list, y, cv_idx, model_name, glm_kwarg_lst, verbose=0, score_method='mse',
                   rows=None, shift_inx=[], fill_value=np.nan, group=None, src=0):
    """`sglm_pp.timeshift_multiple(X0, shift_inx, shift_amt_list)[rows] -> sglm_cv.cv_glm_mult_params(design, y,
    cv_idx, ...)` for ONE session on all GPUs of the process group (NCCL).  Rank `src` passes the host (numpy) or
    device inputs, the other ranks None; every rank gets the reference's result dict (backend/sglm_cv.py:420-426).

      broadcast   base signals X0 [T, P], y and the test-row lists (a few hundred MB; never the 32 GB design)
      gather      every rank builds ITS slice of the design rows locally (lag halo included)
      statistics  row-sharded tcgen05 Gram of the slice; int64 plane Grams all-reduced (exact: the statistics have
                  the bits of the one-GPU run), every rank derives the same centred problems
      fits        models dealt to the ranks by cost; each rank runs its share of the batched plan
      results     one packed all_gather of [coef | intercept | RSS | info]; selection on every rank

    Poisson, Gamma and Tweedie sets (log link) run the batched IRLS of sglm_cv, one batch per distinct power, on the
    rows [g0, g1) of this rank's slice of the design: every cross-row sum of an iteration (objective and gradient
    sums, X'R, the weighted Hessian Gram, the scores) is combined over the ranks (RankComm), so every rank runs every
    log-link model in lock step and holds all their coefficients.  Unlike the Gaussian statistics, the fp64 gradient
    sums are re-associated over the ranks: the log-link results agree with the one-GPU grid to rounding, not to the bit.

    Sets with an l1_ratio (TweedieElasticNet) run in the batch of their power, with the same combined sums.

    rows = (lo, hi): base rows kept after `dropna` (default: the rows without NaN padding).  Folds must be the
    usual complement pairs with duplicate-free test rows (cv_idx_by_*); Gaussian, Poisson, Gamma and Tweedie
    families, mixed in one call."""
    import torch
    import _engine as eng
    import sglm_
    import sglm_cv
    import sglm_pp
    global last_timeline
    dist = _dist()
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    dev = torch.device("cuda", torch.cuda.current_device())
    ev = []

    def mark(name):
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        ev.append((name, e))

    mark("start")
    shifts = [int(a) for a in shift_amt_list]
    smax, smin = max(0, max(shifts)), min(0, min(shifts))
    # ---- source rank: inputs to the device, fold checks; the shapes travel as one small int64 header
    HDR = 72                                                          # T, P, lo, hi, F, ok, then up to 64 fold sizes
    hdr = torch.zeros(HDR, dtype=torch.int64, device=dev)
    if rank == src:
        X0d = eng.device_matrix(X0)
        T, P = X0d.shape
        lo, hi = (smax, T + smin) if rows is None else (int(rows[0]), int(rows[1]))
        n = hi - lo
        yd = eng.device_vector(y)
        if yd.numel() != n:
            raise ValueError(f"Found input variables with inconsistent numbers of samples: [{n}, {yd.numel()}]")
        cv = sglm_cv._normalise_cv_idx(list(cv_idx), n)
        tests = sglm_cv._unique_sorted_rows(cv, n)
        ok = tests is not None and len(cv) <= HDR - 8 and all(len(tr) + len(te) == n for tr, te in cv)
        if ok:
            _, _, _, _, comp = sglm_cv._fold_weights(cv, n)
            ok = bool(np.all(comp))
        head = [T, P, lo, hi, len(cv), int(ok)] + ([int(t.numel()) for t in tests] if ok else [])
        hdr[:len(head)] = torch.tensor(head, dtype=torch.int64)
    mark("prepare")
    dist.broadcast(hdr, src=src, group=group)
    h = hdr.cpu().numpy()
    if not h[5]:
        raise NotImplementedError("cv_grid_strong needs complement train/test folds with duplicate-free test rows "
                                  "(at most 64 folds)")
    T, P, lo, hi, F = (int(v) for v in h[:5])
    n_te = [int(v) for v in h[6:6 + F]]
    n = hi - lo
    if rank != src:
        X0d = torch.empty((T, P), dtype=torch.float64, device=dev)
        yd = torch.empty(n, dtype=torch.float64, device=dev)
        tests = [torch.empty(k, dtype=torch.int64, device=dev) for k in n_te]
    X0d = X0d.contiguous()
    dist.broadcast(X0d, src=src, group=group)
    dist.broadcast(yd, src=src, group=group)
    packed = torch.cat(tests) if F else torch.empty(0, dtype=torch.int64, device=dev)
    dist.broadcast(packed, src=src, group=group)
    tests = list(torch.split(packed, n_te)) if F else []
    mark("broadcast")

    # ---- this rank's rows of the design: valid rows [g0, g1), gathered from the base rows they reach
    g0, g1 = n * rank // world, n * (rank + 1) // world
    src_cols, sh_cols, _ = sglm_pp.build_column_map(P, shift_inx, shifts)
    # ... as a recipe: the statistics come from the base signals (eng.LagRecipe), the slice of the design is only built
    # when a column reads outside the base signals or a log-link family needs it for its GEMMs
    Xd = eng.LagRecipe(X0d, src_cols, sh_cols, lo + g0, lo + g1, fill_value)
    C = Xd.shape[1]
    mark("gather")

    # ---- parameter sets -> estimators (identical on every rank: every raise below happens on every rank)
    entries = []
    for kw in glm_kwarg_lst:
        name = kw.pop('model_name', 'Gaussian')                    # backend/sglm_cv.py:288
        entries.append((name, kw))
    glms, rolls = [], []
    for name, kw in entries:
        rolls.append(int(kw.pop('roll', 0)))                       # backend/sglm_cv.py:95
        glms.append(sglm_.GLM(name, **kw))
        if glms[-1].model.kind not in GAUSSIAN_KINDS + LOG_LINK_KINDS:
            raise NotImplementedError("cv_grid_strong: Gaussian, Poisson, Gamma and Tweedie (log link) families")
    gauss = [i for i, g in enumerate(glms) if g.model.kind in GAUSSIAN_KINDS]
    by_power = {}                                                  # one batch per distinct power, as sglm_cv._cv_batch
    for i, g in enumerate(glms):
        if g.model.kind in LOG_LINK_KINDS:
            by_power.setdefault(1.0 if g.model.kind == "poisson" else g.model.power, []).append(i)
    # ---- this rank's part of every test list (sorted global lists -> local row numbers)
    bounds = torch.tensor([g0, g1], dtype=torch.int64, device=dev)
    local_tests = []
    for t in tests:
        cut = torch.searchsorted(t, bounds).cpu().numpy()
        local_tests.append(t[int(cut[0]):int(cut[1])] - g0)
    comm = RankComm(group)

    def y_columns(rs):
        """The local rows of y and of its rolled copies (rolled over ALL rows), column 0 un-rolled."""
        roll_vals = [0] + sorted({r for r in rs if r % max(n, 1) != 0})
        ycol_of_roll = {r: k for k, r in enumerate(roll_vals)}
        for r in rs:
            if r % max(n, 1) == 0:
                ycol_of_roll[r] = 0
        cols = [yd if k == 0 else eng.roll_vector(yd, int(r)) for k, r in enumerate(roll_vals)]
        return torch.stack([c[g0:g1] for c in cols], dim=1).contiguous(), ycol_of_roll

    out = [None] * len(glms)
    mine = []
    if gauss:
        g_glms, g_rolls = [glms[i] for i in gauss], [rolls[i] for i in gauss]
        Yd, _ = y_columns(g_rolls)
        G = eng.suffstats_tc_sharded(Xd, Yd, [None] + local_tests, comm.all_reduce)
        mark("statistics")

        ses = sglm_cv.GaussianSession.from_statistics(G, n, C, yd, n_te, g_glms, g_rolls, score_method)
        models = ses.model_specs()
        M = len(models)
        owner, _ = deal_models([model_cost(s) for s in models], world)
        owner_lists = [np.flatnonzero(owner == r) for r in range(world)]
        mine = owner_lists[rank]
        mark("problems")
        W, info, status = eng.solve_models([models[i] for i in mine], C)
        mark("fits")
        b_d, rss_full, rss_test, rss_train = ses.score(W, mine)
        n_pad = max(len(o) for o in owner_lists) if M else 0
        mine_pack = pack_results(W[:, :C], b_d, rss_full, rss_test, rss_train, info, status, n_pad)
        gathered = torch.empty((world, n_pad, C + 11), dtype=torch.float64, device=dev)
        dist.all_gather_into_tensor(gathered.reshape(world * n_pad, C + 11), mine_pack, group=group)
        mark("scores+all_gather")
        full = unpack_results(gathered, owner_lists, C)

        n_sets = len(g_glms)
        W3 = full[:, :C].reshape(n_sets, F + 1, C)
        coef_folds = W3[:, :F, :].permute(0, 2, 1).contiguous().cpu().numpy()
        coef_full = W3[:, F, :].contiguous().cpu().numpy()
        tail = full[:, C:].cpu().numpy()
        res = ses.assemble(coef_folds, coef_full, tail[:, 0].copy(), tail[:, 2].copy(), tail[:, 3].copy(),
                           tail[:, 4:10].copy(), tail[:, 10].astype(np.int64))
        for i, r in zip(gauss, res):
            out[i] = r
        mark("download+assemble")
    if by_power:
        # the log-link families: this rank's rows of the design for the two GEMMs of every iteration, its rows of the
        # train / test weights (complement folds: train = 1 - test), the finiteness check combined over the ranks
        Xl = Xd.tensor()
        finite = torch.isfinite(Xl).all().to(torch.int32).reshape(1)
        comm.all_reduce(finite, "min")
        if not bool(finite.item()):
            raise ValueError("Input X contains NaN or infinity.")
        te_w = [eng.index_counts(t, g1 - g0) for t in local_tests]
        RW = torch.stack([1.0 - w for w in te_w] + te_w).contiguous() if F else None
        mark("loglink_design")
        for power, idx in by_power.items():
            l_rolls = [rolls[i] for i in idx]
            Yl, ycol_of_roll = y_columns(l_rolls)
            res = sglm_cv._tweedie_cv(Xl, Yl, ycol_of_roll, RW, F, [glms[i] for i in idx], l_rolls, score_method,
                                      power, comm)
            for i, r in zip(idx, res):
                out[i] = r
            mark(f"loglink_fits_power_{power:g}")
        del Xl, RW
    del Xd
    for (name, kw), r in zip(entries, out):
        r['glm_kwargs'] = kw
    torch.cuda.synchronize()
    last_timeline = {name: float(ev[k - 1][1].elapsed_time(e)) for k, (name, e) in enumerate(ev) if k > 0}
    last_timeline["models_on_this_rank"] = int(len(mine))
    return sglm_cv._select_best([sglm_cv._order_result(r) for r in out], score_method)
