"""Reference numerics for the elastic-net Tweedie tests (TweedieElasticNet), in numpy / scipy: the penalised optimum of

    mean(l(y, eta)) + alpha r |w|_1 + alpha (1 - r)/2 |w|^2,   eta = X w + b,  b unpenalised

with the unit loss l of scikit-learn's HalfTweedieLoss (log link), as L-BFGS-B on split variables w = u - v, u, v >= 0
at a tight gtol, then a few Newton steps on the support it found (smooth there: the sign of w is fixed) to take the
result to rounding level.  Also the KKT residuals of a candidate and the null-model penalty.  A helper of
tests/test_tweedie_enet_args.py and tests/test_gpu_tweedie_enet.py, not a test module itself."""
import numpy as np
from scipy.optimize import minimize

import tweedie_reference as tref


def objective(X, y, w, b, alpha, l1_ratio, power):
    """The penalised mean loss above."""
    eta = X @ w + b
    return float(np.mean(tref.tweedie_terms(eta, y, power)[0]) + alpha * l1_ratio * np.sum(np.abs(w))
                 + 0.5 * alpha * (1.0 - l1_ratio) * (w @ w))


def loss_gradient(X, y, w, b, power):
    """(g, g_b): the gradient of mean(l(y, eta)) in w and in b."""
    d = tref.tweedie_terms(X @ w + b, y, power)[1]
    return X.T @ d / len(y), float(d.mean())


def kkt_residuals(X, y, w, b, alpha, l1_ratio, power, fit_intercept=True):
    """(on-support residual max |g_j + alpha (1-r) w_j + alpha r sign w_j| over w_j != 0, off-support excess
    max(|g_j| - alpha r, 0) over w_j == 0, |g_b| (0 without intercept), g)."""
    g, gb = loss_gradient(X, y, w, b, power)
    nz = w != 0
    on = np.abs(g + alpha * (1.0 - l1_ratio) * w + alpha * l1_ratio * np.sign(w))[nz]
    off = np.maximum(np.abs(g[~nz]) - alpha * l1_ratio, 0.0)
    return (float(on.max()) if on.size else 0.0, float(off.max()) if off.size else 0.0,
            abs(gb) if fit_intercept else 0.0, g)


def alpha_max(X, y, l1_ratio, power, fit_intercept=True):
    """The smallest alpha whose optimum has w = 0: max_j |g_j| / r with g the loss gradient at (w = 0, b = log mean y)
    (b = 0 without an intercept)."""
    b = float(np.log(np.mean(y))) if fit_intercept else 0.0
    g, _ = loss_gradient(X, y, np.zeros(X.shape[1]), b, power)
    return float(np.max(np.abs(g)) / l1_ratio)


def enet_fit(X, y, alpha, l1_ratio, fit_intercept=True, power=1.0, gtol=1e-13):
    """(w, b, f) at the optimum of the objective above."""
    X = np.asarray(X, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64).reshape(-1)
    n, p = X.shape
    a1, a2 = alpha * l1_ratio, alpha * (1.0 - l1_ratio)
    b0 = float(np.log(y.mean())) if fit_intercept else 0.0

    def unpack(z):
        return z[:p] - z[p:2 * p], (z[2 * p] if fit_intercept else 0.0)

    def fun(z):
        w, b = unpack(z)
        terms, d, _ = tref.tweedie_terms(X @ w + b, y, power)
        gw = X.T @ d / n + a2 * w
        f = float(np.mean(terms) + a1 * np.sum(z[:2 * p]) + 0.5 * a2 * (w @ w))
        grad = np.concatenate([gw + a1, -gw + a1] + ([[d.mean()]] if fit_intercept else []))
        return f, grad

    z0 = np.zeros(2 * p + int(fit_intercept))
    if fit_intercept:
        z0[-1] = b0
    bounds = [(0.0, None)] * (2 * p) + ([(None, None)] if fit_intercept else [])
    res = minimize(fun, z0, jac=True, method="L-BFGS-B", bounds=bounds,
                   options=dict(maxiter=50000, maxfun=100000, gtol=gtol, ftol=1e-16, maxcor=50))
    w, b = unpack(res.x)
    w = np.where(np.abs(w) <= 1e-10 * max(1.0, np.max(np.abs(w))), 0.0, w)
    w, b = _polish(X, y, w, b, a1, a2, fit_intercept, power)
    return w, float(b), objective(X, y, w, b, alpha, l1_ratio, power)


def _polish(X, y, w, b, a1, a2, fit_intercept, power, steps=20):
    """Newton steps with step halving on the smooth problem of the support S of w (signs s fixed):
    mean(l) + a1 s'w_S + a2/2 |w_S|^2.  Kept only while the signs hold and the objective does not rise."""
    S = np.flatnonzero(w)
    if len(S) == 0 and not fit_intercept:
        return w, b
    s = np.sign(w[S])
    n = len(y)

    def f_of(wS, b_):
        ww = np.zeros_like(w)
        ww[S] = wS
        return float(np.mean(tref.tweedie_terms(X @ ww + b_, y, power)[0]) + a1 * (s @ wS) + 0.5 * a2 * (wS @ wS))

    XS = X[:, S]
    wS = w[S].copy()
    f = f_of(wS, b)
    for _ in range(steps):
        _, d, v = tref.tweedie_terms(XS @ wS + b, y, power)
        g = XS.T @ d / n + a1 * s + a2 * wS
        H = (XS.T * (v / n)) @ XS + a2 * np.eye(len(S))
        if fit_intercept:
            hb = XS.T @ (v / n)
            H = np.block([[H, hb[:, None]], [hb[None, :], np.array([[v.sum() / n]])]])
            g = np.concatenate([g, [d.mean()]])
        step = np.linalg.solve(H, -g) if len(g) else g
        t = 1.0
        while t > 1e-6:
            wn = wS + t * step[:len(S)]
            bn = b + t * step[-1] if fit_intercept else 0.0
            if np.all(np.sign(wn) == s):
                fn = f_of(wn, bn)
                if fn <= f + 1e-15 * abs(f):
                    break
            t *= 0.5
        else:
            break
        wS, b, f = wn, bn, fn
        if np.max(np.abs(t * step)) <= 1e-15 * max(1.0, np.max(np.abs(wS), initial=0.0)):
            break
    out = np.zeros_like(w)
    out[S] = wS
    return out, b
