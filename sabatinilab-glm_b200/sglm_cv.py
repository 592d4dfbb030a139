"""
sglm_cv — drop-in for the reference module `backend/sglm_cv.py`: cross-validated grid of
penalised GLM fits.  Same entry points and result dictionaries; the execution plan is
B200-native (see _engine.py): the reference runs `len(glm_kwarg_lst) * (n_folds + 1)`
scikit-learn fits one after another from Python threads, copying X[idx_train,:] for
every fold (backend/sglm_cv.py:106-110, :162-170, :180-181); here the whole grid is

    statistics (one pass over X per row set)  ->  ONE batched coordinate-descent launch
    for every ElasticNet/Lasso model + one Cholesky launch per fold for Ridge/OLS  ->
    scores from the statistics,

with identical results (coefficients, per-fold scores, pooled R^2 / MSE, selection).

Reference semantics kept on purpose (results-affecting): `roll` and `model_name` are
popped from the caller's dicts (:95, :288); the full-data refit uses the UN-rolled y
(:181); selection uses strict '>' in list order (:402-415); Ridge alpha is not scaled by
n while ElasticNet's is (backend/sglm.py:102-110).
Not reproduced (crash / hang / waste): the worker-queue hang with fast fits (:22-30,
:169-170) and the discarded PCA + OLS prefit (:275-282).
"""
import itertools

import numpy as np

import _engine as eng
import sglm_


class SGLM_worker():
    """Kept for API compatibility (backend/sglm_cv.py:15-40).  The GPU plan batches the
    work of all workers into single launches, so the queue is drained synchronously."""

    def __init__(self, queue, verbose=0):
        self.queue = queue
        self.verbose = verbose

    def run_single(self):
        while not self.queue.empty():
            glm, args, kwargs = self.queue.get()
            glm.fit_set(*args, **kwargs)
            self.queue.task_done()

    def run_multi(self):
        while not self.queue.empty():
            args, kwargs = self.queue.get()
            cv_glm_single_params(*args, **kwargs)
            self.queue.task_done()


# --------------------------------------------------------------------------- #
# the batched plan
# --------------------------------------------------------------------------- #
def _normalise_cv_idx(cv_idx, T):
    """Fold index lists as the reference uses them (X[idx, :], backend/sglm_cv.py:106-110): boolean masks become
    positions, negative positions wrap, anything outside [-T, T) raises IndexError as numpy does.  Host lists stay
    numpy int64 arrays, CUDA tensors stay on the device (one fused range check for all of them)."""
    import torch
    out, checks = [], []
    for pair in cv_idx:
        norm = []
        for idx in pair:
            if eng.is_torch(idx):
                t = idx.reshape(-1)
                if t.dtype == torch.bool:
                    if t.numel() != T:
                        raise IndexError(f"boolean index did not match indexed array along axis 0; size of axis is {T} "
                                         f"but size of corresponding boolean axis is {t.numel()}")
                    t = torch.nonzero(t).reshape(-1)
                t = t.to(device="cuda", dtype=torch.int64)
                if t.numel():
                    checks.append(((t < -T) | (t >= T)).any())
                norm.append(torch.where(t < 0, t + T, t))
            else:
                a = np.asarray(idx).reshape(-1)
                if a.dtype == bool:
                    if a.shape[0] != T:
                        raise IndexError(f"boolean index did not match indexed array along axis 0; size of axis is {T} "
                                         f"but size of corresponding boolean axis is {a.shape[0]}")
                    a = np.flatnonzero(a)
                a = a.astype(np.int64, copy=False)
                lo_, hi_ = (int(a.min()), int(a.max())) if a.size else (0, 0)
                if lo_ < -T or hi_ >= T:
                    bad = a[(a < -T) | (a >= T)][0]
                    raise IndexError(f"index {int(bad)} is out of bounds for axis 0 with size {T}")
                norm.append(np.where(a < 0, a + T, a) if lo_ < 0 else a)       # the usual lists need no wrap
        out.append(tuple(norm))
    if checks and bool(torch.stack(checks).any().item()):
        raise IndexError(f"index out of bounds for axis 0 with size {T}")
    return out


def _fold_weights(cv_idx, T):
    """Row multiplicities of every train / test index list (X[idx,:] semantics) and whether
    each train set is exactly the complement of its test set (then train = full - test)."""
    import torch
    te = [eng.index_counts(test, T) for (_, test) in cv_idx]
    tr = [eng.index_counts(train, T) for (train, _) in cv_idx]
    n_te = [int(len(test)) for (_, test) in cv_idx]
    n_tr = [int(len(train)) for (train, _) in cv_idx]
    if cv_idx:
        comp = torch.stack([((a + b) == 1.0).all() for a, b in zip(tr, te)]).cpu().numpy()
    else:
        comp = np.zeros(0, dtype=bool)
    return tr, te, n_tr, n_te, comp


def _use_tensor_core_gram(T, C):
    """SGLM_GRAM=dmma|tc overrides; by default the tensor-core path is used once the Gram is
    large enough for its fixed costs (two analysis passes, plan sync) to pay off."""
    import os
    mode = os.environ.get("SGLM_GRAM", "auto")
    if mode == "dmma":
        return False
    if mode == "tc":
        return True
    return T * C * C >= (1 << 33)


def _unique_sorted_rows(cv_idx, T):
    """Sorted, duplicate-free test rows per fold as CUDA int64 tensors, or None when a test
    list repeats rows (then the weighted fp64 path is used).  The lists were normalised by
    _normalise_cv_idx (positions in [0, T))."""
    import torch
    ts = []
    for (_, test) in cv_idx:
        t = test if eng.is_torch(test) else torch.from_numpy(np.ascontiguousarray(test, dtype=np.int64))
        ts.append(t.to(device="cuda", dtype=torch.int64))
    if not ts:
        return []
    # one read-back for all folds: is the list already ascending and duplicate-free (the usual case)?
    asc = torch.stack([(t[1:] > t[:-1]).all() if t.numel() > 1 else torch.ones((), dtype=torch.bool, device="cuda")
                       for t in ts]).cpu().numpy()
    out = []
    for t, ok in zip(ts, asc):
        if ok:
            out.append(t)
            continue
        u = eng.sorted_unique_rows(t, T)
        if u.numel() != t.numel():
            return None
        out.append(u)
    return out


class GaussianSession:
    """One cross-validation problem of Gaussian-family GLMs — (X, y, folds, parameter sets) — cut into the stages
    of the batched plan, so that the stages of SEVERAL problems can be batched (multi-session grids: one
    coordinate-descent launch for all sessions' models) or spread over GPUs (sglm_dist: statistics row-sharded
    and all-reduced, models dealt to ranks):

        build_statistics()  G[s] for s = full data, every test fold (train = full - test), explicit train sets
        model_specs()       one ModelSpec per (parameter set, fold) + per refit, set-major
        score(W, sel)       intercepts and train / test / full RSS of the models `sel` from the statistics
        assemble(...)       the reference's result dicts (backend/sglm_cv.py:188-200)"""

    def __init__(self, Xd, yd, cv_idx, glms, rolls, score_method):
        import torch
        self.Xd, self.yd, self.glms, self.rolls, self.score_method = Xd, yd, glms, rolls, score_method
        self.T, self.C = Xd.shape
        T = self.T
        self.cv_idx = cv_idx
        self.F = len(cv_idx)
        # y columns: column 0 = un-rolled y (refit, backend/sglm_cv.py:181), then one per distinct roll
        roll_vals = [0] + sorted({r for r in rolls if r % max(T, 1) != 0})
        self.ycol_of_roll = {}
        cols = []
        for k, r in enumerate(roll_vals):
            cols.append(yd if k == 0 else eng.roll_vector(yd, int(r)))
            self.ycol_of_roll[r] = k
        for r in rolls:
            if r % max(T, 1) == 0:
                self.ycol_of_roll[r] = 0
        self.Yd = torch.stack(cols, dim=1).contiguous() if len(cols) > 1 else yd.reshape(-1, 1)
        self.n_y = self.Yd.shape[1]
        self.G = None
        self.problems = {}

    @classmethod
    def from_statistics(cls, G, T, C, y_full, n_te, glms, rolls, score_method):
        """A session whose statistics were computed elsewhere (sglm_dist: row-sharded over the GPUs and
        all-reduced): G[0] = all T rows, G[1 + f] = test rows of fold f (n_te[f] of them), every train set the
        complement of its test set.  y_full (CUDA, all T rows) only defines the y columns of the rolls."""
        import torch
        self = cls.__new__(cls)
        self.Xd, self.yd, self.glms, self.rolls, self.score_method = None, y_full, glms, rolls, score_method
        self.T, self.C, self.F = int(T), int(C), len(n_te)
        self.cv_idx = None
        roll_vals = [0] + sorted({r for r in rolls if r % max(self.T, 1) != 0})
        self.roll_vals = roll_vals
        self.ycol_of_roll = {r: k for k, r in enumerate(roll_vals)}
        for r in rolls:
            if r % max(self.T, 1) == 0:
                self.ycol_of_roll[r] = 0
        self.n_y = len(roll_vals)
        self.Yd = None
        self.G, self.problems = G, {}
        self.n_te, self.n_tr = list(n_te), [self.T - n for n in n_te]
        self.extra, self.train_set = [], {f: None for f in range(self.F)}
        self.finite_flag = torch.isfinite(G[0]).all()
        return self

    # ------------------------------------------------------------------ statistics
    def fold_sets(self):
        """Row sets of the statistics: (n_te, n_tr, extra, test_rows | None).  extra = folds whose train rows are
        not the complement of their test rows (they get explicit train statistics)."""
        tr_w, te_w, n_tr, n_te, comp = _fold_weights(self.cv_idx, self.T)
        self.n_te, self.n_tr = n_te, n_tr
        self.extra = [f for f in range(self.F) if not comp[f]]
        self.train_set = {f: (1 + self.F + self.extra.index(f)) if f in self.extra else None for f in range(self.F)}
        return tr_w, te_w

    def build_statistics(self, G=None):
        """set 0 = full data, 1..F = test folds, then explicit train sets.  `G` given: statistics computed
        elsewhere (the row-sharded, all-reduced Gram of sglm_dist)."""
        import torch
        T, C, F = self.T, self.C, self.F
        tr_w, te_w = self.fold_sets()
        if G is None and not self.extra and _use_tensor_core_gram(T, C):
            # 0/1 row sets: tcgen05 int8 digit-plane Gram (exact integer accumulation, fp64 result); a lag design that
            # is still a recipe (eng.LagRecipe) gets its digit planes from the base signals — it is never built
            test_rows = _unique_sorted_rows(self.cv_idx, T)
            if test_rows is not None:
                G, _ = eng.suffstats_tc(self.Xd, self.Yd, [None] + test_rows)
        if G is None and isinstance(self.Xd, eng.LagRecipe):
            self.Xd = self.Xd.tensor()
        if G is None:
            # general row multiplicities: fp64 DMMA Gram with row weights (at most 64 row sets per launch)
            w_rows = [None] + te_w + [tr_w[f] for f in self.extra]
            rows_hint = [T] + self.n_te + [self.n_tr[f] for f in self.extra]
            parts = []
            for c0 in range(0, len(w_rows), 64):
                chunk = w_rows[c0:c0 + 64]
                if len(chunk) == 1 and chunk[0] is None:
                    W = None
                else:
                    W = torch.stack([torch.ones_like(self.yd) if w is None else w for w in chunk]).contiguous()
                parts.append(eng.suffstats(self.Xd, self.Yd, W, rows_hint[c0:c0 + 64]))
            G = parts[0] if len(parts) == 1 else torch.cat(parts, dim=0)
        self.G = G
        self.finite_flag = torch.isfinite(G[0]).all()            # read back together with the results
        return G

    def problem(self, fold, ycol, fi):
        key = (fold, ycol, bool(fi))
        if key not in self.problems:
            G, C, n_y, T = self.G, self.C, self.n_y, self.T
            if fold is None:
                p = eng.center(G[0], None, C, n_y, ycol, fi, n_rows=T)
            elif self.train_set[fold] is None:
                p = eng.center(G[0], G[1 + fold], C, n_y, ycol, fi, n_rows=T - self.n_te[fold])
            else:
                p = eng.center(G[self.train_set[fold]], None, C, n_y, ycol, fi, n_rows=self.n_tr[fold])
            self.problems[key] = p
        return self.problems[key]

    def model_specs(self):
        """ModelSpecs in set-major order: the F fold fits of a set, then its full-data refit."""
        specs, self.owner = [], []            # owner[i] = (param set k, fold f or None)
        for k, (glm, r) in enumerate(zip(self.glms, self.rolls)):
            est = glm.model
            est._check_supported()
            for f in list(range(self.F)) + [None]:
                p = self.problem(f, self.ycol_of_roll[r] if f is not None else 0, est.fit_intercept)
                specs.append(est._spec(p))    # no device read-back: row counts are known on the host
                self.owner.append((k, f))
        self.models = specs
        return specs

    # ------------------------------------------------------------------ scores from the statistics
    def score(self, Wd, sel=None):
        """Intercepts and residual sums of squares of the models `sel` (indices into model_specs(); default all),
        whose coefficients are the rows of Wd: RSS(set) = V' G[set] V.  Returns device tensors
        (b, rss_full, rss_test, rss_train), each [len(sel)]."""
        import torch
        sel = list(range(len(self.models))) if sel is None else list(sel)
        models = [self.models[i] for i in sel]
        b_d, V = eng.finalize(Wd, self.C, self.n_y, models)
        M = len(models)
        fold_of = np.array([-1 if self.owner[i][1] is None else self.owner[i][1] for i in sel])
        rss_full = eng.quadform(self.G[0], V)
        rss_test = torch.zeros(M, dtype=torch.float64, device="cuda")
        rss_train = rss_full.clone()
        for f in range(self.F):
            pick = np.flatnonzero(fold_of == f)
            if len(pick) == 0:
                continue
            pick_t = eng._dev(pick, np.int64)
            Vf = V.index_select(0, pick_t)
            q_te = eng.quadform(self.G[1 + f], Vf)
            rss_test.index_copy_(0, pick_t, q_te)
            if self.train_set[f] is None:
                rss_train.index_copy_(0, pick_t, rss_full.index_select(0, pick_t) - q_te)
            else:
                rss_train.index_copy_(0, pick_t, eng.quadform(self.G[self.train_set[f]], Vf))
        return b_d, rss_full, rss_test, rss_train

    def moments(self):
        """[set, (y cols | 1), (y cols | 1)] block of the statistics on the host (n, sum y, y'y of every row set)."""
        C, n_y = self.C, self.n_y
        return self.G[:, C:, C:C + n_y + 1].cpu().numpy()

    # ------------------------------------------------------------------ result dicts
    def assemble(self, coef_folds, coef_full, icpt, rss_test_h, rss_train_h, info, status, Gy=None):
        """coef_folds [set][C][F], coef_full [set][C], icpt / rss_* / info / status per model (set-major), all on
        the host -> the reference's per-set result dicts."""
        if not bool(self.finite_flag.item()):
            raise ValueError("Input contains NaN, infinity or a value too large for dtype('float64').")
        glms, rolls, F, n_y = self.glms, self.rolls, self.F, self.n_y
        ycol_of_roll, train_set, score_method = self.ycol_of_roll, self.train_set, self.score_method
        n_sets_k = len(glms)
        Gy = self.moments() if Gy is None else Gy

        def set_moments(s, ycol):
            return Gy[s, n_y, n_y], Gy[s, ycol, n_y], Gy[s, ycol, ycol]

        # per-fold moments of every y column (vectorised over the folds; the loop below runs once per set)
        mom = {}
        for ycol in sorted(set(ycol_of_roll.values())):
            n_f = np.array([set_moments(1 + f, ycol)[0] for f in range(F)])
            sy_f = np.array([set_moments(1 + f, ycol)[1] for f in range(F)])
            yy_f = np.array([set_moments(1 + f, ycol)[2] for f in range(F)])
            n_t, sy_t, yy_t = np.zeros(F), np.zeros(F), np.zeros(F)
            n0, sy0, yy0 = set_moments(0, ycol)
            for f in range(F):
                if train_set[f] is None:
                    n_t[f], sy_t[f], yy_t[f] = n0 - n_f[f], sy0 - sy_f[f], yy0 - yy_f[f]
                else:
                    n_t[f], sy_t[f], yy_t[f] = set_moments(train_set[f], ycol)
            with np.errstate(divide='ignore', invalid='ignore'):
                tss_f = np.where(n_f > 0, yy_f - sy_f * sy_f / n_f, 0.0)
                tss_t = np.where(n_t > 0, yy_t - sy_t * sy_t / n_t, 0.0)
            mom[ycol] = (n_f, n_t, tss_f, tss_t)

        def r2_vec(rss, tss):
            with np.errstate(divide='ignore', invalid='ignore'):
                return np.where(tss <= 0.0, np.where(rss == 0.0, 1.0, 0.0), 1.0 - rss / np.where(tss <= 0.0, 1.0, tss))

        # scores of every (set, fold) at once
        ycols = np.array([ycol_of_roll[r] for r in rolls], dtype=np.int64)
        fi = np.array([bool(g.model.fit_intercept) for g in glms])
        rte = np.maximum(rss_test_h.reshape(n_sets_k, F + 1)[:, :F], 0.0)
        rtr = np.maximum(rss_train_h.reshape(n_sets_k, F + 1)[:, :F], 0.0)
        icpt2 = icpt.reshape(n_sets_k, F + 1)
        n_f = np.stack([mom[c][0] for c in ycols]) if n_sets_k else np.zeros((0, F))
        n_t = np.stack([mom[c][1] for c in ycols]) if n_sets_k else np.zeros((0, F))
        tss_f = np.stack([mom[c][2] for c in ycols]) if n_sets_k else np.zeros((0, F))
        tss_t = np.stack([mom[c][3] for c in ycols]) if n_sets_k else np.zeros((0, F))
        if score_method == 'r2':
            S_tr, S_te = r2_vec(rtr, tss_t), r2_vec(rte, tss_f)
        else:
            with np.errstate(divide='ignore', invalid='ignore'):
                S_tr, S_te = -rtr / n_t, -rte / n_f
        rss_pool_a = np.zeros(n_sets_k)
        tss_pool_a = np.zeros(n_sets_k)
        n_pool_a = np.zeros(n_sets_k)
        for f in range(F):                                   # left-to-right, as the reference accumulates fold by fold
            rss_pool_a += rte[:, f]
            tss_pool_a += np.maximum(tss_f[:, f], 0.0)
            n_pool_a += n_f[:, f]
        with np.errstate(divide='ignore', invalid='ignore'):
            mean_tr = S_tr.mean(axis=1) if F else np.full(n_sets_k, np.nan)
            mean_te = S_te.mean(axis=1) if F else np.full(n_sets_k, np.nan)
            std_te = S_te.std(axis=1) if F else np.full(n_sets_k, np.nan)

        results = []
        for k, glm in enumerate(glms):
            base = k * (F + 1)
            rss_pool, tss_pool, n_pool = rss_pool_a[k], tss_pool_a[k], n_pool_a[k]
            i_full = base + F
            _set_fitted(glm, coef_full[k], icpt[i_full], info[i_full], status[i_full])
            results.append({
                'cv_coefs': coef_folds[k],
                'cv_intercepts': icpt2[k, :F].copy() if fi[k] else np.zeros(F),
                'cv_scores_train': S_tr[k].copy(),
                'cv_scores_test': S_te[k].copy(),
                'cv_mean_score_train': mean_tr[k],
                'cv_mean_score': mean_te[k],
                'cv_std_score': std_te[k],
                'cv_R2_score': 0 if tss_pool == 0 else 1 - rss_pool / tss_pool,      # sglm.calc_R2
                'cv_mse_score': rss_pool / n_pool if n_pool else np.nan,
                'model': glm,
                '_fit_info': {'cd_info': info[base:base + F + 1], 'status': status[base:base + F + 1]},
            })
            bad = status[base:base + F + 1]
            if np.any(bad == 2):
                raise np.linalg.LinAlgError("Matrix is singular: X'X + alpha*I is not positive definite")
        return results

    def download_coefficients(self, Wd, ready=None):
        """Coefficients leave the device already in the layout of the result dicts: [set][C][F] for the folds
        (cv_coefs is C x F, backend/sglm_cv.py:98) and [set][C] for the refits — one transposition on the device
        instead of one per parameter set on the host.  With `ready` (an event recorded when Wd was complete) the
        transposition and the copies run on a side stream, next to whatever the caller has queued on the current
        stream since (the score kernels)."""
        import torch
        C, F = self.C, self.F
        n_sets_k = len(self.glms)

        def fetch():
            W3 = Wd[:, :C].reshape(n_sets_k, F + 1, C)
            return (W3[:, :F, :].permute(0, 2, 1).contiguous().cpu().numpy(),         # [set][C][F]
                    W3[:, F, :].contiguous().cpu().numpy())                            # [set][C]
        if ready is None:
            return fetch()
        side = eng._side_stream(200)
        side.wait_event(ready)
        with torch.cuda.stream(side):
            out = fetch()                                   # .cpu() waits for the side stream only
        Wd.record_stream(side)
        return out

    def download_and_assemble(self, Wd, b_d, rss_test, rss_train, info, status, coefs=None):
        coef_folds, coef_full = self.download_coefficients(Wd) if coefs is None else coefs
        return self.assemble(coef_folds, coef_full, b_d.cpu().numpy(), rss_test.cpu().numpy(),
                             rss_train.cpu().numpy(), info, status)


def _gaussian_grid(Xd, yd, cv_idx, glms, rolls, score_method):
    """Fit every (param set, fold) + every full-data refit of Gaussian-family GLMs.
    glms: list of sglm_.GLM objects (already dispatched to an estimator class)."""
    ses = GaussianSession(Xd, yd, cv_idx, glms, rolls, score_method)
    ses.build_statistics()
    models = ses.model_specs()
    import torch
    Wd, info, status = eng.solve_models(models, ses.C)
    ready = torch.cuda.Event()
    ready.record()
    b_d, _, rss_test, rss_train = ses.score(Wd)              # queued; the coefficients travel meanwhile
    coefs = ses.download_coefficients(Wd, ready)
    return ses.download_and_assemble(Wd, b_d, rss_test, rss_train, info, status, coefs)


def cv_glm_mult_params_sessions(sessions, model_name, glm_kwarg_lst, verbose=0, score_method='mse'):
    """Extension (BASELINE configs[4], SURVEY.md §8e): the same parameter grid on SEVERAL independent sessions
    — `sessions` = [(X, y, cv_idx), ...] with the same number of design columns — as ONE batched plan: the
    statistics of every session, then one coordinate-descent launch (and one Cholesky launch per problem) over
    the models of all sessions, so that the heavy-tailed models of one session overlap the light ones of the
    others.  Returns [cv_glm_mult_params-style dict per session]; each equals what a separate call returns."""
    per_session = []
    all_models = []
    for (X, y, cv_idx) in sessions:
        entries = []
        for glm_kwargs in glm_kwarg_lst:
            kw = dict(glm_kwargs)
            name = kw.pop('model_name', model_name if model_name is not None else 'Gaussian')
            entries.append((name, kw))
        Xd, yd = eng.device_design(X), eng.device_vector(y)
        if Xd.shape[0] != yd.shape[0]:
            raise ValueError(f"Found input variables with inconsistent numbers of samples: [{Xd.shape[0]}, {yd.shape[0]}]")
        cv = _normalise_cv_idx(list(cv_idx), Xd.shape[0])
        glms, rolls = [], []
        for name, kw in entries:
            rolls.append(int(kw.pop('roll', 0)))
            glms.append(sglm_.GLM(name, **kw))
            if glms[-1].model.kind not in ("ols", "ridge", "lasso", "enet"):
                raise NotImplementedError("cv_glm_mult_params_sessions batches the Gaussian family")
        ses = GaussianSession(Xd, yd, cv, glms, rolls, score_method)
        ses.build_statistics()
        models = ses.model_specs()
        per_session.append((ses, entries, len(all_models), len(models)))
        all_models.extend(models)
    C = per_session[0][0].C if per_session else 0
    if any(ses.C != C for ses, _, _, _ in per_session):
        raise ValueError("cv_glm_mult_params_sessions: every session must have the same number of design columns")
    Wd, info, status = eng.solve_models(all_models, C)
    out = []
    for ses, entries, m0, m in per_session:
        Ws = Wd[m0:m0 + m]
        b_d, _, rss_test, rss_train = ses.score(Ws)
        res = ses.download_and_assemble(Ws, b_d, rss_test, rss_train, info[m0:m0 + m], status[m0:m0 + m])
        for (name, kw), r in zip(entries, res):
            r['glm_kwargs'] = kw
        out.append(_select_best([_order_result(r) for r in res], score_method))
    return out


def _r2(rss, tss):
    if tss <= 0.0:
        return 1.0 if rss == 0.0 else 0.0
    return 1.0 - rss / tss


def _set_fitted(glm, coef, intercept, info, status):
    est = glm.model
    est.coef_ = np.array(coef, dtype=np.float64)
    est.intercept_ = float(intercept) if est.fit_intercept else 0.0
    est.n_features_in_ = len(coef)
    if est.kind in ("enet", "lasso"):
        est.dual_gap_ = float(info[0])
        est.n_iter_ = int(info[2])
    glm.coef_ = est.coef_
    glm.beta_ = glm.coef_
    glm.intercept_ = est.intercept_
    glm.beta0_ = glm.intercept_


def _poisson_grid(Xd, yd, cv_idx, glms, rolls, score_method, power=1.0):
    """Poisson family (backend/sglm.py:112-115), or the Tweedie family of `power` > 1 (Gamma: power 2, :112-117):
    every (parameter set, fold) fit and every refit of the grid as ONE batched Newton-type iteration
    (`_engine.tweedie_grid_batched`: X is read once per iteration for all models, one tcgen05 weighted Gram per fold
    as the shared approximate Hessian, exact gradients), then one batched scoring pass for the train / test sums of
    every fold model.  'r2' scores are the family's D^2; -MSE and the pooled cv_R2_score / cv_mse_score are
    residual-based."""
    import torch
    T, C = Xd.shape
    F = len(cv_idx)
    _, te_w, _, n_te, _ = _fold_weights(cv_idx, T)
    tr_w = [eng.index_counts(train, T) for (train, _) in cv_idx]
    RW = torch.stack(tr_w + te_w).contiguous() if F else None             # rows 0..F-1 train, F..2F-1 test weights
    if not bool(torch.isfinite(Xd).all().item()):
        raise ValueError("Input X contains NaN or infinity.")
    roll_vals = [0] + sorted({r for r in rolls if r % max(T, 1) != 0})
    ycol_of_roll = {r: k for k, r in enumerate(roll_vals)}
    for r in rolls:
        if r % max(T, 1) == 0:
            ycol_of_roll[r] = 0
    Yd = torch.stack([yd if k == 0 else eng.roll_vector(yd, int(r)) for k, r in enumerate(roll_vals)], dim=1).contiguous()
    return _tweedie_cv(Xd, Yd, ycol_of_roll, RW, F, glms, rolls, score_method, power)


def _tweedie_cv(Xd, Yd, ycol_of_roll, RW, F, glms, rolls, score_method, power, comm=None):
    """The batched fits and scores of _poisson_grid from its inputs: the response columns Yd (one per distinct roll,
    column 0 un-rolled), the row weights RW (rows 0..F-1 train, F..2F-1 test).  comm: the rows are sharded over
    processes (sglm_dist.cv_grid_strong; see _engine.tweedie_grid_batched) — every process returns the same results."""
    C = Xd.shape[1]
    models, ycol, rw_a, rw_b = [], [], [], []
    for glm, r in zip(glms, rolls):
        est = glm.model
        est._check_family()
        l1_ratio = est.l1_ratio if est.kind == "tweedie_enet" else 0.0
        for f in range(F):
            models.append(eng.PoissonModel(est.alpha, est.fit_intercept, rw=f, ycol=ycol_of_roll[r],
                                           max_iter=est.max_iter, tol=est.tol, l1_ratio=l1_ratio))
            ycol.append(ycol_of_roll[r]); rw_a.append(f); rw_b.append(F + f)
        models.append(eng.PoissonModel(est.alpha, est.fit_intercept, rw=-1, ycol=0, max_iter=est.max_iter, tol=est.tol,
                                       l1_ratio=l1_ratio))
        ycol.append(0); rw_a.append(-1); rw_b.append(-2)          # the refit uses the UN-rolled y (backend/sglm_cv.py:181)
    Wd, bd, n_it, status = eng.tweedie_grid_batched(Xd, Yd, models, RW, power, comm)
    sums = eng.tweedie_scores_batched(Xd, Yd, Wd, bd, ycol, rw_a, rw_b, RW, power, comm)
    W_h, b_h = Wd.cpu().numpy(), bd.cpu().numpy()
    results = []
    for k, glm in enumerate(glms):
        est = glm.model
        base = k * (F + 1)
        cv_coefs = np.ascontiguousarray(W_h[base:base + F].T) if F else np.zeros((C, 0))
        cv_intercepts = b_h[base:base + F].copy() if est.fit_intercept else np.zeros(F)
        s_tr, s_te = np.zeros(F), np.zeros(F)
        rss_pool = tss_pool = n_pool = 0.0
        for f in range(F):
            st, se = sums[base + f, 0], sums[base + f, 1]
            if score_method == 'r2':
                s_tr[f], s_te[f] = eng.tweedie_d2_from_sums(st, power), eng.tweedie_d2_from_sums(se, power)
            else:
                s_tr[f], s_te[f] = -st[1] / st[0], -se[1] / se[0]
            rss_pool += se[1]
            tss_pool += se[3] - se[2] * se[2] / se[0]
            n_pool += se[0]
        w, b = W_h[base + F].copy(), float(b_h[base + F]) if est.fit_intercept else 0.0
        est.coef_, est.intercept_, est.n_iter_ = w, b, int(n_it[base + F])
        est.n_features_in_ = C
        glm.coef_ = glm.beta_ = w
        glm.intercept_ = glm.beta0_ = b
        results.append({
            'cv_coefs': cv_coefs, 'cv_intercepts': cv_intercepts,
            'cv_scores_train': s_tr, 'cv_scores_test': s_te,
            'cv_mean_score_train': np.mean(s_tr) if F else np.nan, 'cv_mean_score': np.mean(s_te) if F else np.nan,
            'cv_std_score': np.std(s_te) if F else np.nan,
            'cv_R2_score': 0 if tss_pool == 0 else 1 - rss_pool / tss_pool,
            'cv_mse_score': rss_pool / n_pool if n_pool else np.nan,
            'model': glm,
            '_fit_info': {'n_iter': n_it[base:base + F + 1], 'status': status[base:base + F + 1]},
        })
    return results


def _cv_batch(X, y, cv_idx, entries, beta_, beta0_, score_method):
    Xd = eng.device_design(X)          # a contiguous device-resident lag design stays a recipe (never built)
    yd = eng.device_vector(y)
    if Xd.shape[0] != yd.shape[0]:
        raise ValueError(f"Found input variables with inconsistent numbers of samples: [{Xd.shape[0]}, {yd.shape[0]}]")
    cv_idx = _normalise_cv_idx(list(cv_idx), Xd.shape[0])
    glms, rolls = [], []
    for model_name, kw in entries:
        rolls.append(int(kw.pop('roll', 0)))                          # backend/sglm_cv.py:95
        glms.append(sglm_.GLM(model_name, beta0_=beta0_, beta_=beta_, **kw))   # refit object (:180)
    out = [None] * len(entries)
    gauss = [i for i, g in enumerate(glms) if g.model.kind in ("ols", "ridge", "lasso", "enet")]
    # the log-link families: one batch per distinct power, Poisson (power 1) first; elastic-net sets join the batch of
    # their power
    by_power = {}
    for i, g in enumerate(glms):
        if g.model.kind in ("poisson", "tweedie", "tweedie_enet"):
            by_power.setdefault(1.0 if g.model.kind == "poisson" else g.model.power, []).append(i)
    if gauss:
        res = _gaussian_grid(Xd, yd, cv_idx, [glms[i] for i in gauss], [rolls[i] for i in gauss], score_method)
        for i, r in zip(gauss, res):
            out[i] = r
    if by_power and isinstance(Xd, eng.LagRecipe):
        Xd = Xd.tensor()
    for power, idx in by_power.items():
        res = _poisson_grid(Xd, yd, cv_idx, [glms[i] for i in idx], [rolls[i] for i in idx], score_method, power)
        for i, r in zip(idx, res):
            out[i] = r
    for (model_name, kw), r in zip(entries, out):
        r['glm_kwargs'] = kw
    return out


def _order_result(r):
    keys = ['cv_coefs', 'cv_intercepts', 'cv_scores_train', 'cv_scores_test', 'cv_mean_score_train',
            'cv_mean_score', 'cv_std_score', 'cv_R2_score', 'cv_mse_score', 'glm_kwargs', 'model']
    out = {k: r[k] for k in keys}
    for k in r:
        if k not in out:
            out[k] = r[k]
    return out


def cv_glm_single_params(X, y, cv_idx, model_name, glm_kwargs, verbose=0, resp_list=[], beta_=None, beta0_=None,
                         score_method='mse'):
    """Cross-validation for one parameter set: F fold fits + one full-data refit.
    Returns the reference's dict (backend/sglm_cv.py:188-200) and appends it to resp_list."""
    ret_dict = _order_result(_cv_batch(X, y, cv_idx, [(model_name, glm_kwargs)], beta_, beta0_, score_method)[0])
    if verbose > 0:
        print('Completing arguments:', glm_kwargs)
        print(f"{glm_kwargs}\n> cv_mean_score_train: {ret_dict['cv_mean_score_train']}\n> cv_R2_score: "
              f"{ret_dict['cv_R2_score']}\n> cv_mean_score: {ret_dict['cv_mean_score']}")
    resp_list.append(ret_dict)
    return ret_dict


def cv_glm_mult_params(X, y, cv_idx, model_name, glm_kwarg_lst, verbose=0, score_method='mse'):
    """Cross-validation over a list of parameter sets; picks the best by `score_method`
    ('r2' -> pooled cv_R2_score, 'mse' -> cv_mean_score) with the reference's strict '>' in
    list order (backend/sglm_cv.py:210-428)."""
    entries = []
    for glm_kwargs in glm_kwarg_lst:
        if verbose > 0:
            print(glm_kwargs)
        name = glm_kwargs.pop('model_name', 'Gaussian')               # backend/sglm_cv.py:288
        entries.append((name, glm_kwargs))
    resp = [_order_result(r) for r in _cv_batch(X, y, cv_idx, entries, None, None, score_method)]
    if verbose > 0:
        for r in resp:
            print(f"{r['glm_kwargs']}\n> cv_mean_score_train: {r['cv_mean_score_train']}\n> cv_R2_score: "
                  f"{r['cv_R2_score']}\n> cv_mean_score: {r['cv_mean_score']}")
    return _select_best(resp, score_method)


def _select_best(resp, score_method):
    """The reference's selection: strict '>' in list order (backend/sglm_cv.py:402-415)."""
    best_score = -np.inf
    best_params = None
    for cv_result in resp:
        if (score_method == 'r2' and cv_result['cv_R2_score'] > best_score):
            best_score = cv_result['cv_R2_score']
            best_score_std = cv_result['cv_std_score']
            best_params = cv_result['glm_kwargs']
            best_model = cv_result['model']
        elif (score_method == 'mse' and cv_result['cv_mean_score'] > best_score):
            best_score = cv_result['cv_mean_score']
            best_score_std = cv_result['cv_std_score']
            best_params = cv_result['glm_kwargs']
            best_model = cv_result['model']
    return {
        'best_score': best_score,
        'best_score_std': best_score_std,
        'best_params': best_params,
        'best_model': best_model,
        'full_cv_results': resp,
    }


def generate_mult_params(kwarg_lists, kwargs=None):
    """Every combination of the listed values merged over the fixed kwargs: fixed keys first,
    then `kwarg_lists` keys in insertion order, last key varying fastest
    (backend/sglm_cv.py:476-496)."""
    keys = list(kwarg_lists)
    combos = itertools.product(*[list(kwarg_lists[k]) for k in keys])
    out = []
    for combo in combos:
        d = dict(kwargs) if kwargs else {}
        for k, v in zip(keys, combo):
            d[k] = v
        out.append(d)
    return out
