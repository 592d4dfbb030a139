"""TweedieElasticNet on the GPU (Poisson, Gamma, Tweedie with an L1 + L2 penalty, log link): single fits against the
CPU reference optimum (tests/tweedie_enet_reference.py) with their KKT conditions and supports, the null model above
alpha_max, warm starts, CV grids that mix elastic-net and ridge sets against per-fold single fits and host-computed
scores, the strong-scaled path (a single-rank comm, and 2 ranks sharing one GPU over gloo), one fit at the
tensor-core Hessian size, and the proximal-Newton step entry point (sglm_pb_step_enet_f64) on a tiny batch."""
import ctypes
import os
import socket
import sys

import numpy as np
import pytest

from conftest import PKG, ROOT, coef_rel_err
import tweedie_enet_reference as eref
import tweedie_reference as tref

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
if not torch.cuda.is_available():
    pytest.skip("needs a CUDA device", allow_module_level=True)

import synth_data  # noqa: E402
import _engine as eng  # noqa: E402
import _sglm_native as nat  # noqa: E402
import sglm  # noqa: E402
import sglm_cv  # noqa: E402
from _estimators import TweedieElasticNet  # noqa: E402

EPS_KKT = 1e-7          # KKT residuals of a converged fit: the outer step bound is 1e-8 relative, times the curvature


def _problem(n, p, seed, power):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((n, p))
    X[:, 1] = X[:, 0] + 0.3 * rng.standard_normal(n)            # correlated columns
    X[:, 2] += 0.5                                               # a column with a non-zero mean
    beta = np.zeros(p)
    beta[:4] = [0.4, -0.3, 0.2, 0.1]
    mu = np.exp(0.6 * (X @ beta) - 0.5)
    y = rng.poisson(mu).astype(np.float64) if power == 1 else synth_data.tweedie_draw(mu, seed, power)
    return X, y


def _kkt_ok(X, y, w, b, alpha, r, power, fit_intercept, eps=EPS_KKT):
    on, off, gb, g = eref.kkt_residuals(X, y, w, b, alpha, r, power, fit_intercept)
    return on <= eps and off <= eps and gb <= eps, (on, off, gb)


@pytest.mark.parametrize("power", [1.0, 1.5, 2.0, 3.0])
@pytest.mark.parametrize("l1_ratio", [0.1, 0.5, 1.0])
@pytest.mark.parametrize("fit_intercept", [True, False])
def test_single_fit_vs_reference(power, l1_ratio, fit_intercept):
    X, y = _problem(3000, 12, 11, power)
    alpha = 0.15 * eref.alpha_max(X, y, l1_ratio, power, fit_intercept)
    w_ref, b_ref, f_ref = eref.enet_fit(X, y, alpha, l1_ratio, fit_intercept, power)
    est = TweedieElasticNet(power=power, alpha=alpha, l1_ratio=l1_ratio, fit_intercept=fit_intercept, tol=1e-10)
    est.fit(X, y)
    w, b = est.coef_, est.intercept_
    f = eref.objective(X, y, w, b, alpha, l1_ratio, power)
    assert f <= f_ref + 1e-12 * abs(f), (f, f_ref)
    assert coef_rel_err(w, w_ref) <= 1e-6, coef_rel_err(w, w_ref)
    ok, res = _kkt_ok(X, y, w, b, alpha, l1_ratio, power, fit_intercept)
    assert ok, res
    # the support, outside coordinates whose |g_j| is within EPS_KKT of alpha r (either side is optimal there)
    g, _ = eref.loss_gradient(X, y, w_ref, b_ref, power)
    clear = np.abs(np.abs(g) - alpha * l1_ratio) > EPS_KKT
    assert np.array_equal((w != 0)[clear], (w_ref != 0)[clear])
    assert 0 < np.count_nonzero(w) < len(w)
    # score / predict: the family's D^2 and exp(X w + b)
    mu = np.exp(X @ w + b)
    assert abs(est.score(X, y) - tref.tweedie_d2(y, mu, power)) <= 1e-10
    assert np.max(np.abs(est.predict(X) - mu)) <= 1e-12 * np.max(mu)
    # warm start from the optimum (the reference's, at rounding level — as tests/test_gpu_tweedie.py does; the fit
    # above is only held to its step bound, 1e-10 * max(1, |w|_inf), which is looser than 1e-9 |w|_inf for |w| < 1):
    # stops at once, at the same coefficients
    warm = TweedieElasticNet(power=power, alpha=alpha, l1_ratio=l1_ratio, fit_intercept=fit_intercept, tol=1e-10,
                             warm_start=True)
    warm.coef_, warm.intercept_ = w_ref.copy(), b_ref
    warm.fit(X, y)
    assert warm.n_iter_ <= 3 and coef_rel_err(warm.coef_, w_ref) <= 1e-9, (warm.n_iter_, coef_rel_err(warm.coef_, w_ref))
    assert abs(warm.intercept_ - b_ref) <= 1e-9 * max(1.0, abs(b_ref))


@pytest.mark.parametrize("power", [1.0, 1.5, 2.0, 3.0])
def test_null_model_above_alpha_max(power):
    X, y = _problem(3000, 12, 13, power)
    for r in (0.5, 1.0):
        a = 1.000001 * eref.alpha_max(X, y, r, power, True)
        g = sglm.GLM("Tweedie", power=power, alpha=a, l1_ratio=r) if power not in (1.0, 2.0) else \
            sglm.GLM("Poisson" if power == 1.0 else "Gamma", alpha=a, l1_ratio=r)
        assert isinstance(g.model, TweedieElasticNet)
        g.fit(X, y)
        assert np.all(g.coef_ == 0.0)
        b0 = np.log(y.mean())
        assert abs(g.intercept_ - b0) <= 1e-14 * abs(b0), (g.intercept_, b0)


def test_sessions_still_reject_log_link_sets():
    X, y = _problem(400, 4, 3, 1.0)
    cv = [(np.arange(0, 300), np.arange(300, 400))]
    with pytest.raises(NotImplementedError):
        sglm_cv.cv_glm_mult_params_sessions([(X, y, cv)], "Poisson", [dict(alpha=.1, l1_ratio=.5)])


# --------------------------------------------------------------------------- CV grids
def _grid_data():
    X, _ = _problem(4000, 10, 21, 1.0)
    rng = np.random.default_rng(21)
    mu = np.exp(0.3 * X[:, 0] - 0.2 * X[:, 3] - 0.5)
    y = synth_data.tweedie_draw(mu, 21, 2.0)                    # y > 0: valid for Poisson and Gamma
    folds = synth_data.synth_folds(len(y), 3, 21, group=100)
    del rng
    return X, y, folds


def _grid(X, y):
    am = eref.alpha_max(X, y, 0.5, 1.0)
    sets = []
    for r in (0.0, 0.5, 1.0):
        for k in (0.05, 0.3, 1.2):
            a = k * (am * 0.5 if r == 0 else am * 0.5 / r)      # alpha_max(r) = alpha_max(0.5) * 0.5 / r
            sets.append(dict(alpha=float(a), l1_ratio=r, model_name="Poisson", max_iter=200, tol=1e-10))
    sets.append(dict(alpha=float(0.3 * eref.alpha_max(X, y, 0.5, 2.0)), l1_ratio=0.5, model_name="Gamma", max_iter=200,
                     tol=1e-10))
    return sets


def _power_of(s):
    return 2.0 if s["model_name"] == "Gamma" else 1.0


def _host_scores(X, y, folds, w_cols, b_f, power, score_method):
    tr_s, te_s, rss, tss, n_te = [], [], 0.0, 0.0, 0
    for f, (tr, te) in enumerate(folds):
        w, b = w_cols[:, f], b_f[f]
        out = []
        for rows in (tr, te):
            mu = np.exp(X[rows] @ w + b)
            out.append(tref.tweedie_d2(y[rows], mu, power) if score_method == "r2" else -np.mean((y[rows] - mu) ** 2))
        tr_s.append(out[0]); te_s.append(out[1])
        r = y[te] - np.exp(X[te] @ w + b)
        rss += r @ r
        tss += np.sum((y[te] - y[te].mean()) ** 2)
        n_te += len(te)
    return np.array(tr_s), np.array(te_s), 1.0 - rss / tss, rss / n_te


@pytest.mark.parametrize("score_method", ["r2", "mse"])
def test_cv_grid_vs_single_fits_and_host_scores(score_method):
    X, y, folds = _grid_data()
    sets = _grid(X, y)
    res = sglm_cv.cv_glm_mult_params(X, y, folds, "Poisson", [dict(s) for s in sets], score_method=score_method)
    full = res["full_cv_results"]
    assert len(full) == len(sets)
    keys = []
    for s, r in zip(sets, full):
        power = _power_of(s)
        if s["l1_ratio"] != 0:
            assert isinstance(r["model"].model, TweedieElasticNet)
            for f, (tr, _) in enumerate(folds):
                one = TweedieElasticNet(power=power, alpha=s["alpha"], l1_ratio=s["l1_ratio"], max_iter=200, tol=1e-10)
                one.fit(X[tr], y[tr])
                assert coef_rel_err(r["cv_coefs"][:, f], one.coef_) <= 1e-7, (s, f)
                assert abs(r["cv_intercepts"][f] - one.intercept_) <= 1e-7 * max(1.0, abs(one.intercept_))
        tr_s, te_s, r2, mse = _host_scores(X, y, folds, r["cv_coefs"], r["cv_intercepts"], power, score_method)
        assert np.max(np.abs(r["cv_scores_train"] - tr_s)) <= 1e-10
        assert np.max(np.abs(r["cv_scores_test"] - te_s)) <= 1e-10
        assert abs(r["cv_R2_score"] - r2) <= 1e-10 and abs(r["cv_mse_score"] - mse) <= 1e-10
        keys.append(r2 if score_method == "r2" else np.mean(te_s))
    best, best_k = -np.inf, None
    for k, v in enumerate(keys):
        if v > best:
            best, best_k = v, k
    assert res["best_params"] == full[best_k]["glm_kwargs"]
    # the ridge sets of the mixed batch agree with the same sets run alone
    ridge = [s for s in sets if s["l1_ratio"] == 0]
    alone = sglm_cv.cv_glm_mult_params(X, y, folds, "Poisson", [dict(s) for s in ridge], score_method=score_method)
    mixed = [r for s, r in zip(sets, full) if s["l1_ratio"] == 0]
    for a, b in zip(mixed, alone["full_cv_results"]):
        for j in range(len(folds)):
            assert coef_rel_err(a["cv_coefs"][:, j], b["cv_coefs"][:, j]) <= 1e-9
        assert np.max(np.abs(a["cv_intercepts"] - b["cv_intercepts"])) <= 1e-9
        assert coef_rel_err(a["model"].coef_, b["model"].coef_) <= 1e-9


def test_cv_grid_reports_inner_sweeps():
    X, y, folds = _grid_data()
    sets = [s for s in _grid(X, y) if s["model_name"] == "Poisson"]
    sglm_cv.cv_glm_mult_params(X, y, folds, "Poisson", [dict(s) for s in sets], score_method="r2")
    d = eng.last_poisson_batch[0]
    assert d["enet_models"] == 6 * (len(folds) + 1) and d["inner_sweeps"] > 0 and d["rounds"] >= 1


# --------------------------------------------------------------------------- tensor-core Hessian size
def test_fit_at_tensor_core_hessian_size():
    T, C = 70_000, 1000                                          # T C^2 >= 2^36: the tcgen05 weighted Gram
    assert eng._poisson_tc(T, C)
    rng = np.random.default_rng(5)
    X = torch.randn(T, C, dtype=torch.float64, device="cuda", generator=torch.Generator("cuda").manual_seed(5))
    beta = torch.zeros(C, dtype=torch.float64, device="cuda")
    beta[:20] = torch.from_numpy(rng.uniform(-0.1, 0.1, 20)).cuda()
    y = torch.poisson(torch.exp(X @ beta - 0.5), generator=torch.Generator("cuda").manual_seed(6))
    r = 0.5
    b0 = float(torch.log(y.mean()))
    g0 = X.t() @ (torch.exp(torch.full_like(y, b0)) - y) / T
    alpha = 0.2 * float(g0.abs().max()) / r
    est = TweedieElasticNet(power=1, alpha=alpha, l1_ratio=r, tol=1e-10).fit(X, y)
    assert eng.last_poisson_batch[0]["tensor_core_hessian"]
    w = torch.from_numpy(est.coef_).cuda()
    d = torch.exp(X @ w + est.intercept_) - y
    g = (X.t() @ d / T).cpu().numpy()
    wn = est.coef_
    nz = wn != 0
    assert 0 < nz.sum() < C
    assert np.max(np.abs(g + alpha * (1 - r) * wn + alpha * r * np.sign(wn))[nz]) <= EPS_KKT
    assert np.max(np.abs(g[~nz])) <= alpha * r + EPS_KKT
    assert abs(float(d.mean())) <= EPS_KKT


# --------------------------------------------------------------------------- strong path
class _OneRank:
    """comm of a single process: nothing to exchange, the partials pass through the fixed-order sum."""

    def all_reduce(self, t, op):
        assert op in ("max", "min", "sum")

    def combine(self, t):
        return eng.reduce_parts(t.reshape(-1).contiguous(), 1).reshape(t.shape)


@pytest.mark.parametrize("use_tc", [True, False])
@pytest.mark.parametrize("power", [1.0, 1.5])
def test_single_rank_comm_is_bit_identical_with_l1_models(power, use_tc):
    X, y, folds = _grid_data()
    T = len(y)
    Xd = torch.from_numpy(X).cuda()
    Yd = torch.from_numpy(y).cuda()[:, None].contiguous()
    RW = torch.stack([eng.index_counts(a, T) for a, _ in folds]).contiguous()
    models = []
    for alpha, r in ((1e-3, 0.0), (2e-2, 0.5), (5e-2, 1.0), (1e-2, 0.1)):
        for f in range(len(folds)):
            models.append(eng.PoissonModel(alpha, True, rw=f, tol=1e-10, l1_ratio=r))
        models.append(eng.PoissonModel(alpha, True, rw=-1, tol=1e-10, l1_ratio=r))
    old = eng.POISSON_TC
    eng.POISSON_TC = use_tc
    try:
        W0, b0, it0, st0 = eng.tweedie_grid_batched(Xd, Yd, models, RW, power)
        d0 = dict(eng.last_poisson_batch[0])
        W1, b1, it1, st1 = eng.tweedie_grid_batched(Xd, Yd, models, RW, power, comm=_OneRank())
        d1 = dict(eng.last_poisson_batch[0])
    finally:
        eng.POISSON_TC = old
    assert d0["tensor_core_hessian"] == use_tc and d0["inner_sweeps"] > 0
    assert torch.equal(W0, W1) and torch.equal(b0, b1)
    assert np.array_equal(it0, it1) and np.array_equal(st0, st1) and d0 == d1
    assert set(np.unique(st0)) == {1}


SHIFTS = [0] + [s for s in range(-3, 5) if s != 0]


def _strong_inputs():
    from oracle import sglm_oracle as orc
    X0 = synth_data.synth_base(6000, 4, 21)
    d = orc.timeshift_multiple(X0, shift_amt_list=SHIFTS)[4:-3]
    y = synth_data.synth_response_tweedie(d, synth_data.synth_kernels(4, SHIFTS, 21), 21, 2.0)
    folds = synth_data.synth_folds(d.shape[0], 4, 21, group=150)
    grid = ([dict(model_name="Poisson", alpha=a, l1_ratio=r, tol=1e-10) for r in (0.5, 1.0) for a in (2e-3, 2e-2)] +
            [dict(model_name="Poisson", alpha=1e-2, tol=1e-10), dict(model_name="Gamma", alpha=1e-2, l1_ratio=0.5, tol=1e-10),
             dict(alpha=1e-2, l1_ratio=0.5, max_iter=1000)])
    return X0, d, y, folds, grid


def _worker(rank, world, port, ret):
    for p in (ROOT, PKG):
        if p not in sys.path:
            sys.path.insert(0, p)
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import sglm_cv as cv
    import sglm_dist
    X0, d, y, folds, grid = _strong_inputs()
    res = sglm_dist.cv_grid_strong(X0 if rank == 0 else None, SHIFTS, y if rank == 0 else None,
                                   folds if rank == 0 else None, "Gaussian", [dict(g) for g in grid], score_method="r2")
    rec = [repr(res["best_params"])] + [np.concatenate([r["cv_coefs"].ravel(), r["cv_intercepts"], r["model"].coef_,
                                                        [r["model"].intercept_, r["cv_R2_score"]]]).tobytes()
                                        for r in res["full_cv_results"]]
    mine = [None] * world
    dist.all_gather_object(mine, rec)
    report = {"ranks_identical": all(m == mine[0] for m in mine)}
    if rank == 0:
        one = cv.cv_glm_mult_params(d, y, folds, "Gaussian", [dict(g) for g in grid], score_method="r2")
        report["best_params"] = (res["best_params"], one["best_params"])
        worst = 0.0
        for a, b, g in zip(res["full_cv_results"], one["full_cv_results"], grid):
            if g.get("model_name", "Gaussian") == "Gaussian":
                continue
            for j in range(a["cv_coefs"].shape[1]):
                worst = max(worst, coef_rel_err(a["cv_coefs"][:, j], b["cv_coefs"][:, j]))
            worst = max(worst, coef_rel_err(a["model"].coef_, b["model"].coef_),
                        float(np.max(np.abs(a["cv_intercepts"] - b["cv_intercepts"]))),
                        abs(a["model"].intercept_ - b["model"].intercept_))
            for k in ("cv_scores_train", "cv_scores_test", "cv_R2_score", "cv_mse_score"):
                worst = max(worst, float(np.max(np.abs(np.subtract(a[k], b[k])))))
        report["worst"] = worst
    ret[rank] = report
    dist.barrier()
    dist.destroy_process_group()


def test_strong_grid_two_ranks_sharing_one_gpu():
    import time
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    mgr = mp.Manager()
    try:
        ret = mgr.dict()
        ctx = mp.start_processes(_worker, args=(2, port, ret), nprocs=2, join=False, start_method="spawn")
        deadline = time.monotonic() + 600
        try:
            while not ctx.join(timeout=5):
                if time.monotonic() > deadline:
                    raise TimeoutError("cv_grid_strong over 2 ranks did not finish in 600 s")
        finally:
            for p in ctx.processes:
                if p.is_alive():
                    p.terminate()
                p.join()
        out = dict(ret)
    finally:
        mgr.shutdown()
    assert sorted(out) == [0, 1]
    assert out[0]["ranks_identical"] and out[1]["ranks_identical"]
    got, want = out[0]["best_params"]
    assert got == want
    print(f"2 ranks (gloo, one GPU): worst difference to one GPU {out[0]['worst']:.3e}")
    assert out[0]["worst"] <= 1e-9


# --------------------------------------------------------------------------- the step entry point
def _dev(a, dtype=torch.float64):
    return torch.from_numpy(np.ascontiguousarray(a)).to(device="cuda", dtype=dtype)


@pytest.mark.parametrize("C", [7, 40, 300])
def test_pb_step_enet_objective_halving_and_inner_kkt(C):
    """Models: 0 ridge (a chord step), 1 and 2 elastic net with a step, 3 elastic net whose L1 term alone makes the
    objective worse than the previous one (halving), 4 elastic net with a borrowed Hessian (hscale != 1)."""
    rng = np.random.default_rng(C)
    B, ldw, ldq, ldb = 5, eng._round_up(C, 2), eng._round_up(C, 8), 64
    A = rng.standard_normal((C, C))
    Q = A @ A.T / C + 0.3 * np.eye(C)
    xbar = rng.uniform(-0.3, 0.3, C)
    h11 = 120.0
    r = np.array([0.0, 0.5, 1.0, 0.3, 0.7])
    alpha = np.array([0.05, 0.2, 0.1, 0.2, 0.3])
    n_tot = rng.uniform(100.0, 300.0, B)
    hscale = np.array([1.0, 1.0, 1.0, 1.0, 1.7])
    W = np.zeros((B, ldw))
    W[:, :C] = rng.uniform(-0.5, 0.5, (B, C)) * (rng.uniform(size=(B, C)) < 0.5)
    Wp = np.zeros((B, ldw))
    Wp[:, :C] = rng.uniform(-0.5, 0.5, (B, C))
    sums = np.zeros((B, 4))
    sums[:, 0] = rng.uniform(50.0, 500.0, B)
    sums[:, 3] = rng.normal(0.0, 2.0, B)
    ww = np.sum(W[:, :C] ** 2, axis=1)
    w1 = np.sum(np.abs(W[:, :C]), axis=1)
    f_ridge = sums[:, 0] / n_tot + 0.5 * (alpha * (1 - r)) * ww
    f_full = f_ridge + alpha * r * w1
    fprev = f_full + 1.0
    fprev[3] = 0.5 * (f_ridge[3] + f_full[3])                    # worse only through the L1 term
    Gw = np.zeros((C, ldb))
    Gw[:, :B] = rng.normal(0.0, 5.0, (C, B))
    d = {k: _dev(v) for k, v in dict(W=W, Wprev=Wp, b=rng.uniform(-1, 1, B), bprev=rng.uniform(-1, 1, B), fprev=fprev,
                                     last_step=np.full(B, 0.5), ratio_out=np.full(B, 0.7), alpha=alpha, n_tot=n_tot,
                                     tol=np.full(B, 1e-4), sums=sums, Gw=Gw, hscale=hscale).items()}
    d["Wnew"] = torch.zeros((B, ldw), dtype=torch.float64, device="cuda")
    d["rhs"] = torch.zeros((B, ldw), dtype=torch.float64, device="cuda")
    d["fcur"] = torch.zeros(B, dtype=torch.float64, device="cuda")
    d["step_out"] = torch.zeros(B, dtype=torch.float64, device="cuda")
    for k, v in dict(halv=np.zeros(B), n_iter=np.full(B, 2), status=np.zeros(B), flag=np.zeros(B), has_prev=np.ones(B),
                     fit_icpt=np.ones(B), max_iter=np.full(B, 100), hess_id=np.zeros(B)).items():
        d[k] = _dev(v.astype(np.int32), torch.int32)
    Qd = torch.zeros((C, ldq), dtype=torch.float64, device="cuda")
    Qd[:, :C] = _dev(Q)
    xb = _dev(xbar)
    d["HQ"] = _dev(np.array([Qd.data_ptr()], np.int64), torch.int64)
    d["Hxbar"] = _dev(np.array([xb.data_ptr()], np.int64), torch.int64)
    d["Hh11"] = _dev(np.array([h11]))
    shift = alpha * (1 - r) * n_tot                              # the factors of (Q + alpha (1 - r) n I)
    an = _dev(shift)
    wb = nat.lib().sglm_ridge_workspace_bytes(C, ldq, B)
    work = torch.empty(wb // 8, dtype=torch.float64, device="cuda")
    Wtmp = torch.empty((B, ldw), dtype=torch.float64, device="cuda")
    st = torch.empty(B, dtype=torch.int32, device="cuda")
    qc = torch.zeros(C, dtype=torch.float64, device="cuda")
    eng.call("sglm_ridge_solve_f64", eng.ptr(Qd), ldq, eng.ptr(qc), C, eng.ptr(an), B, eng.ptr(Wtmp), ldw, eng.ptr(st),
             eng.ptr(work), wb, eng.stream_ptr())
    L_of = _dev(np.array([work.data_ptr() + k * (C + 1) * ldq * 8 for k in range(B)], np.int64), torch.int64)
    order = ["W", "Wprev", "Wnew", "rhs", "b", "bprev", "fprev", "fcur", "last_step", "step_out", "ratio_out", "halv",
             "n_iter", "status", "flag", "has_prev", "alpha", "n_tot", "tol", "fit_icpt", "max_iter", "hess_id", "HQ",
             "Hxbar", "Hh11", "sums", "Gw", "hscale"]
    words = [d[k].data_ptr() for k in order] + [ldw, ldq, ldb, C | (B << 32)]
    assert len(words) == nat.lib().sglm_pb_state_words()
    state = np.array(words, dtype=np.uint64)
    l1r = _dev(r)
    enet = _dev(np.array([1, 2, 3, 4], np.int32), torch.int32)
    ws = torch.empty(nat.lib().sglm_pb_enet_workspace_bytes(C, ldw, 4) // 8 + 1, dtype=torch.float64, device="cuda")
    info = torch.zeros((4, 6), dtype=torch.float64, device="cuda")
    eng.call("sglm_pb_step_enet_f64", state.ctypes.data_as(ctypes.c_void_p), eng.ptr(L_of), eng.ptr(l1r), eng.ptr(enet),
             4, eng.ptr(ws), ws.numel() * 8, eng.ptr(info), eng.stream_ptr())
    torch.cuda.synchronize()
    o = {k: v.cpu().numpy() for k, v in d.items()}
    inf = info.cpu().numpy()
    assert list(o["flag"]) == [1, 1, 1, 2, 1]
    # the objective of the stepping models (fcur) has the L1 term; model 3 was halved because of it
    for k in (0, 1, 2, 4):
        assert abs(o["fcur"][k] - f_full[k]) <= 1e-13 * abs(f_full[k]), (k, o["fcur"][k], f_full[k])
    assert np.array_equal(o["W"][3], 0.5 * (W[3] + Wp[3])) and o["halv"][3] == 1
    assert inf[2, 2] == 0.0 and np.all(inf[[0, 1, 3], 2] >= 1)    # no inner solve for the halving model
    # the inner solve's output (now w) satisfies the KKT conditions of the inner quadratic model
    for k in (1, 2, 4):
        q = o["rhs"][k, :C]
        l1 = alpha[k] * r[k] * n_tot[k] / hscale[k]
        l2 = alpha[k] * (1 - r[k]) * n_tot[k] / hscale[k]
        w = o["W"][k, :C]
        grad = Q @ w - q + l2 * w
        scale = max(1.0, np.max(np.abs(q)))
        nz = w != 0
        assert np.all(np.abs(grad + l1 * np.sign(w))[nz] <= 1e-10 * scale), k
        assert np.all(np.abs(grad[~nz]) <= l1 + 1e-10 * scale), k
    # the ridge model took the chord step: (Q + alpha n I) w_new = rhs
    w0 = o["W"][0, :C]
    assert np.max(np.abs((Q + shift[0] * np.eye(C)) @ w0 - o["rhs"][0, :C])) <= 1e-10 * max(1.0, np.max(np.abs(o["rhs"][0])))
