"""
Seeded synthetic "photometry-shaped" inputs (SURVEY.md §8d) shared by tests, the oracle and
bench.py.  Neutral utility: neither product code nor oracle.  Shapes follow the reference's
drivers: sparse 0/1 event indicators (er_refactored_from_scratch_cleanup.py:203-222), a few
real-valued z-scored AR(1) signals and one within-trial ramp (pp_design_mat.py:171); smooth
exponentially decaying kernels; Gaussian response with AR(1) noise scaled to R^2 ~ 0.3, a
spike-count-like Poisson response, or a Gamma / compound Poisson-Gamma / inverse Gaussian one; GroupShuffleSplit-style folds over 1000-row trials
(backend/sglm_pp.py:262-263).
"""
import numpy as np


def synth_base(T, P, seed, frac_real=0.2):
    """Base predictors X0[T,P]: sparse 0/1 event indicators + z-scored AR(1) + one ramp."""
    rng = np.random.default_rng(seed)
    X0 = np.empty((T, P), dtype=np.float64)
    n_real = max(1, int(round(P * frac_real)))
    for p in range(P):
        if p < P - n_real:
            X0[:, p] = (rng.random(T) < rng.uniform(0.01, 0.03)).astype(np.float64)
        elif p == P - 1:
            X0[:, p] = (np.arange(T) % 1000) / 1000.0
        else:
            from scipy.signal import lfilter
            e = rng.standard_normal(T)
            a = lfilter([1.0], [1.0, -0.95], e)
            X0[:, p] = (a - a.mean()) / a.std()
    return X0


def synth_kernels(P, shifts, seed):
    rng = np.random.default_rng(seed + 7)
    L = len(shifts)
    beta = np.zeros((L, P))
    for p in range(P):
        if rng.random() < 0.3:
            continue
        beta[:, p] = np.exp(-np.abs(np.asarray(shifts)) / 8.0) * rng.standard_normal(L)
    return beta.reshape(-1)


def synth_response(Xd, beta, seed, poisson=False):
    rng = np.random.default_rng(seed + 13)
    from scipy.signal import lfilter
    s = Xd @ beta
    if poisson:
        z = (s - s.mean()) / (s.std() + 1e-300)
        return rng.poisson(np.exp(0.3 * z - 1.0)).astype(np.float64)
    e = lfilter([1.0], [1.0, -0.95], rng.standard_normal(len(s)))
    e = e / e.std() * s.std() * np.sqrt(0.7 / 0.3)
    y = s + e
    return (y - y.mean()) / y.std()


def synth_response_tweedie(Xd, beta, seed, power):
    """Response of the Tweedie family of `power` with log link and mean mu = exp(0.3 z(X beta) - 1), as the
    Poisson response: power 2 Gamma (shape 2), 1 < power < 2 compound Poisson-Gamma with dispersion 1 (exact
    zeros), power 3 inverse Gaussian (numpy Wald, dispersion 1)."""
    s = Xd @ beta
    z = (s - s.mean()) / (s.std() + 1e-300)
    return tweedie_draw(np.exp(0.3 * z - 1.0), seed, power)


def tweedie_draw(mu, seed, power):
    """One draw per mean mu of the distributions of synth_response_tweedie."""
    rng = np.random.default_rng(seed + 17)
    mu = np.asarray(mu, dtype=np.float64)
    if power == 2:
        return rng.gamma(2.0, mu / 2.0)
    if power == 3:
        return rng.wald(mu, 1.0)
    if 1 < power < 2:
        # N ~ Poisson(mu^(2-p) / (2-p)) events, each Gamma(shape (2-p)/(p-1), scale (p-1) mu^(p-1))
        n = rng.poisson(mu ** (2.0 - power) / (2.0 - power))
        shape = n * (2.0 - power) / (power - 1.0)
        y = np.zeros_like(mu)
        pos = n > 0
        y[pos] = rng.gamma(shape[pos], (power - 1.0) * mu[pos] ** (power - 1.0))
        return y
    raise ValueError(f"no synthetic Tweedie response for power={power} (1 < power < 2, 2 or 3)")


def synth_folds(T, n_folds, seed, group=1000, test_size=0.2):
    """GroupShuffleSplit over trial ids arange(T)//group (sglm_pp.py:262-263), restated
    with a seeded Generator so that it needs no sklearn on the bench path."""
    rng = np.random.default_rng(seed + 29)
    groups = np.arange(T) // group
    n_groups = int(groups.max()) + 1
    n_test = max(1, int(np.ceil(test_size * n_groups)))
    out = []
    for _ in range(n_folds):
        perm = rng.permutation(n_groups)
        is_test = np.zeros(n_groups, dtype=bool)
        is_test[perm[:n_test]] = True
        m = is_test[groups]
        out.append((np.flatnonzero(~m), np.flatnonzero(m)))
    return out
