"""Reference numerics for the Gamma / Tweedie (power > 1, log link) tests, in numpy: the unit terms of scikit-learn's
HalfTweedieLoss, the penalised optimum by Fisher scoring, D^2, and the reference's CV loop (backend/sglm_cv.py:42-428)
for parameter sets whose model_name is 'Gamma' or 'Tweedie'; every other family goes to the oracle's restatement.
A helper of tests/test_tweedie_oracle.py and tests/test_gpu_tweedie.py, not a test module itself."""
import numpy as np

from oracle import sglm_oracle as orc


def tweedie_terms(eta, y, power):
    """Unit loss, its derivative in eta and the Fisher weight of sklearn's HalfTweedieLoss with log link."""
    if power == 1:
        mu = np.exp(eta)
        return mu - y * eta, mu - y, mu
    if power == 2:
        y_mu = y * np.exp(-eta)
        return eta + y_mu, 1.0 - y_mu, np.ones_like(eta)
    mu, mu1 = np.exp(eta), np.exp((1.0 - power) * eta)
    mu2 = mu * mu1
    return mu2 / (2.0 - power) - y * mu1 / (1.0 - power), mu1 * (mu - y), mu2


def tweedie_fit(X, y, alpha=1.0, fit_intercept=True, power=2.0, max_iter=1000, tol=1e-12):
    """argmin mean(l(y, eta)) + alpha/2 ||w||^2, eta = Xw + b, with the unit loss l of sklearn's HalfTweedieLoss
    (log link; power 1 Poisson, 2 Gamma, other p: mu^(2-p)/(2-p) - y mu^(1-p)/(1-p); intercept un-penalised; start
    at w = 0, b = log(mean y)).  Fisher scoring (weights mu^(2-p)) with step halving, to a gradient below `tol` or a
    full step below 1e-13 relative (Fisher scoring converges linearly; the objective then changes within rounding, so
    the sufficient-decrease test allows a few ulps of it)."""
    X = np.asarray(X, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64).reshape(-1)
    n, p = X.shape
    w = np.zeros(p)
    b = float(np.log(y.mean())) if fit_intercept else 0.0

    def objective(w_, b_):
        return float(np.mean(tweedie_terms(X @ w_ + b_, y, power)[0]) + 0.5 * alpha * (w_ @ w_))

    f = objective(w, b)
    it = 0
    for it in range(1, max_iter + 1):
        _, d, v = tweedie_terms(X @ w + b, y, power)
        gw = X.T @ (d / n) + alpha * w
        H = (X.T * (v / n)) @ X
        H.flat[:: p + 1] += alpha
        if fit_intercept:
            hb = X.T @ (v / n)
            Hf = np.empty((p + 1, p + 1))
            Hf[:p, :p] = H
            Hf[:p, p] = hb
            Hf[p, :p] = hb
            Hf[p, p] = v.sum() / n
            g = np.concatenate([gw, [d.sum() / n]])
        else:
            Hf, g = H, gw
        if np.max(np.abs(g)) <= tol:
            break
        step = np.linalg.solve(Hf, -g)
        t = 1.0
        while True:
            w_new = w + t * step[:p]
            b_new = b + t * step[p] if fit_intercept else 0.0
            f_new = objective(w_new, b_new)
            if f_new <= f + 1e-4 * t * (g @ step) + 1e-15 * abs(f) or t < 1e-10:
                break
            t *= 0.5
        w, b, f = w_new, b_new, f_new
        if t == 1.0 and np.max(np.abs(step)) <= 1e-13 * max(1.0, np.max(np.abs(w))):
            break
    return w, float(b), dict(n_iter=it)


def tweedie_d2(y, mu, power):
    """D^2 = 1 - dev(y, mu)/dev(y, mean y) with the Tweedie unit deviance of `power` (sklearn
    d2_tweedie_score; TweedieRegressor.score)."""
    if power == 1:
        return orc.poisson_d2(y, mu)
    y = np.asarray(y, dtype=np.float64)
    p = float(power)

    def dev(m):
        if p == 2:
            return float(np.mean(2.0 * (np.log(m / y) + y / m - 1.0)))
        return float(np.mean(2.0 * (y ** (2.0 - p) / ((1.0 - p) * (2.0 - p)) - y * m ** (1.0 - p) / (1.0 - p)
                                    + m ** (2.0 - p) / (2.0 - p))))

    return 1.0 - dev(np.asarray(mu, dtype=np.float64)) / dev(np.full_like(y, y.mean()))


def _power(model_name, kw):
    return 2.0 if model_name == "Gamma" else float(kw.get("power", 0.0))


def _fit(X, y, model_name, kw):
    """(coef, intercept) of one Gamma / Tweedie fit at the optimum (TweedieRegressor keywords)."""
    return tweedie_fit(X, y, kw.get("alpha", 1.0), kw.get("fit_intercept", True), _power(model_name, kw))[:2]


def cv_glm_single_params(X, y, cv_idx, model_name, glm_kwargs, score_method="mse"):
    """orc.cv_glm_single_params for model_name 'Gamma' / 'Tweedie': `roll` popped, fold fits on X[idx], the family's
    D^2 ('r2') or -MSE per fold, pooled R^2 / MSE from the test residuals, full-data refit on the un-rolled y."""
    if model_name not in ("Gamma", "Tweedie"):
        return orc.cv_glm_single_params(X, y, cv_idx, model_name, glm_kwargs, score_method)
    power = _power(model_name, glm_kwargs)
    roll = glm_kwargs.pop("roll", 0)
    y = np.asarray(y, dtype=np.float64).reshape(-1)
    y_rolled = np.roll(y, roll)
    F = len(cv_idx)
    cv_coefs, cv_intercepts = np.zeros((X.shape[1], F)), np.zeros(F)
    tr, te = np.zeros(F), np.zeros(F)
    resids, mean_resids = [], []

    def score(w, b, Xs, ys):
        mu = np.exp(Xs @ w + b)
        return tweedie_d2(ys, mu, power) if score_method == "r2" else -np.mean((ys - mu) ** 2)
    for k, (itr, ite) in enumerate(cv_idx):
        w, b = _fit(X[itr], y_rolled[itr], model_name, glm_kwargs)
        cv_coefs[:, k], cv_intercepts[k] = w, b
        tr[k], te[k] = score(w, b, X[itr], y_rolled[itr]), score(w, b, X[ite], y_rolled[ite])
        resids.append(y_rolled[ite] - np.exp(X[ite] @ w + b))
        mean_resids.append(y_rolled[ite] - y_rolled[ite].mean())
    w, b = _fit(X, y, model_name, glm_kwargs)
    return {"cv_coefs": cv_coefs, "cv_intercepts": cv_intercepts, "cv_scores_train": tr, "cv_scores_test": te,
            "cv_mean_score_train": np.mean(tr), "cv_mean_score": np.mean(te), "cv_std_score": np.std(te),
            "cv_R2_score": orc.calc_R2(np.concatenate(resids), np.concatenate(mean_resids)),
            "cv_mse_score": np.mean(np.square(np.concatenate(resids))), "glm_kwargs": glm_kwargs,
            "model": {"coef_": w, "intercept_": b}}


def cv_glm_mult_params(X, y, cv_idx, glm_kwarg_lst, score_method="mse"):
    """orc.cv_glm_mult_params with Gamma / Tweedie sets allowed: model_name popped from each set (default
    'Gaussian'), strict '>' selection in list order.  The refit of every result is returned as `model_coef` /
    `model_intercept`."""
    resp = []
    for kw in glm_kwarg_lst:
        name = kw.pop("model_name", "Gaussian")
        r = cv_glm_single_params(X, y, cv_idx, name, kw, score_method)
        m = r["model"]
        r["model_coef"], r["model_intercept"] = (m["coef_"], m["intercept_"]) if isinstance(m, dict) else (m.coef_, m.intercept_)
        resp.append(r)
    best_score, best = -np.inf, None
    for r in resp:
        s = r["cv_R2_score"] if score_method == "r2" else r["cv_mean_score"]
        if s > best_score:
            best_score, best = s, r
    return {"best_score": best_score, "best_params": best["glm_kwargs"], "full_cv_results": resp}
