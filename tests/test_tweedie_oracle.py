"""Gamma / Tweedie (log link) without a GPU: the Fisher-scoring optimum of tests/tweedie_reference.py against
scikit-learn's newton-cholesky TweedieRegressor, the D^2 restatements against sklearn.metrics.d2_tweedie_score,
argument checks of the power-taking ABI entry points, and the estimator's family validation."""
import ctypes
import warnings

import numpy as np
import pytest

from conftest import coef_rel_err
from oracle import sglm_oracle as orc
import tweedie_reference as tref

import synth_data
import _engine as eng
import _sglm_native as nat
import sglm


def _design(seed=11, T=3000, P=5):
    shifts = [0] + [s for s in range(-4, 4) if s != 0]
    X0 = synth_data.synth_base(T, P, seed)
    Xd = orc.timeshift_multiple(X0, shift_amt_list=shifts)
    Xd = Xd[~np.isnan(Xd).any(axis=1)]
    return Xd, synth_data.synth_kernels(P, shifts, seed)


def _objective(X, y, w, b, alpha, power):
    return float(np.mean(tref.tweedie_terms(X @ w + b, y, power)[0]) + 0.5 * alpha * (w @ w))


@pytest.mark.parametrize("power", [1.5, 2.0, 3.0])
def test_reference_tweedie_fit_vs_sklearn_newton_cholesky(power):
    from sklearn.linear_model import TweedieRegressor
    Xd, beta = _design()
    y = synth_data.synth_response_tweedie(Xd, beta, 11, power)
    n = len(y)
    for fit_intercept in (True, False):
        for alpha in (1e-3, 0.1):
            w, b, _ = tref.tweedie_fit(Xd, y, alpha, fit_intercept, power)
            with warnings.catch_warnings(record=True) as caught:
                warnings.simplefilter("always")
                ref = TweedieRegressor(power=power, alpha=alpha, fit_intercept=fit_intercept, solver="newton-cholesky",
                                       tol=1e-12, max_iter=1000).fit(Xd, y)
            fell_back = any("NewtonCholeskySolver" in str(c.message) for c in caught)
            if not fell_back:
                assert coef_rel_err(w, ref.coef_) < 1e-8, (power, fit_intercept, alpha)
                assert abs(b - ref.intercept_) < 1e-8
            else:
                # scikit-learn's Newton step met an indefinite pointwise Hessian (power > 2 without intercept) and
                # handed over to L-BFGS, which stops short: the reference must be at least as good and stationary
                d = tref.tweedie_terms(Xd @ w + b, y, power)[1]
                assert np.max(np.abs(Xd.T @ (d / n) + alpha * w)) < 1e-10
                assert _objective(Xd, y, w, b, alpha, power) <= _objective(Xd, y, ref.coef_, ref.intercept_, alpha,
                                                                            power) + 1e-14


@pytest.mark.parametrize("power", [1.0, 1.5, 2.0, 3.0])
def test_tweedie_d2_vs_sklearn_and_from_sums(power):
    """tref.tweedie_d2 against d2_tweedie_score, and the engine's D^2 from the fused score sums (computed here in numpy
    with the kernel's slot layout) against both."""
    from sklearn.metrics import d2_tweedie_score
    rng = np.random.default_rng(3)
    mu = np.exp(rng.normal(-1.0, 0.4, 5000))
    y = synth_data.tweedie_draw(mu, 5, power) if power != 1.0 else rng.poisson(mu).astype(np.float64)
    pred = mu * np.exp(rng.normal(0.0, 0.1, len(mu)))
    want = d2_tweedie_score(y, pred, power=power)
    assert abs(tref.tweedie_d2(y, pred, power) - want) < 1e-12
    eta, r = np.log(pred), y - pred
    if power == 1.0:
        s456 = [np.sum(y * eta), np.sum(pred), np.sum(np.where(y > 0, y * np.log(np.where(y > 0, y, 1.0)), 0.0))]
    elif power == 2.0:
        s456 = [np.sum(eta), np.sum(y / pred), np.sum(np.log(y))]
    else:
        s456 = [np.sum(y * pred ** (1 - power)), np.sum(pred ** (2 - power)), np.sum(y ** (2 - power))]
    s = np.array([len(y), np.sum(r * r), np.sum(y), np.sum(y * y)] + s456 + [np.sum(r)])
    assert abs(eng.tweedie_d2_from_sums(s, power) - want) < 1e-12


def test_synthetic_tweedie_responses():
    Xd, beta = _design()
    y15 = synth_data.synth_response_tweedie(Xd, beta, 11, 1.5)
    assert y15.min() == 0.0 and 0.05 < np.mean(y15 == 0) < 0.9          # compound Poisson-Gamma: exact zeros
    for p in (2.0, 3.0):
        y = synth_data.synth_response_tweedie(Xd, beta, 11, p)
        assert y.min() > 0 and abs(y.mean() - np.exp(-1.0)) < 0.1
    with pytest.raises(ValueError):
        synth_data.tweedie_draw(np.ones(3), 0, 2.5)


def test_glm_abi_entry_points_validate_before_cuda():
    """Shape, null-pointer and power checks of the power-taking entry points run before any CUDA call."""
    lib = nat.lib()
    p = ctypes.c_void_p(64)        # never dereferenced: every call below fails its argument checks first
    ws = nat.lib().sglm_score_workspace_bytes()
    # bad shape
    assert lib.sglm_score_glm_f64(p, 4, p, None, 10, 8, p, p, 2.0, None, p, p, None) == -2
    assert lib.sglm_glm_irls_prepare_f64(p, 8, p, None, -1, 8, p, p, 2.0, p, p, p, p, None) == -2
    assert lib.sglm_glm_epilogue_f64(p, 64, 65, 100, p, 1, p, None, 0, p, None, p, None, 2.0, 0, p, p, 1 << 30, None) == -2
    assert b"bad shape" in lib.sglm_last_error()
    # null pointers
    assert lib.sglm_score_glm_f64(None, 8, p, None, 10, 8, p, p, 2.0, None, p, p, None) == -1
    assert lib.sglm_glm_irls_prepare_f64(p, 8, p, None, 10, 8, p, p, 2.0, None, p, p, p, None) == -1
    assert lib.sglm_glm_epilogue_f64(p, 64, 8, 100, p, 1, p, None, 0, None, None, p, None, 2.0, 0, p, p, 1 << 30, None) == -1
    assert lib.sglm_glm_epilogue_f64(p, 64, 8, 100, p, 1, p, None, 0, p, None, p, None, 2.0, 1, p, p, 1 << 30, None) == -1
    # unsupported powers: <= 0, between 0 and 1, NaN
    for power in (0.0, -1.0, 0.5, 0.999, float("nan")):
        assert lib.sglm_score_glm_f64(p, 8, p, None, 10, 8, p, p, power, None, p, p, None) == -6, power
        assert b"power" in lib.sglm_last_error()
        assert lib.sglm_glm_irls_prepare_f64(p, 8, p, None, 10, 8, p, p, power, p, p, p, p, None) == -6, power
        assert lib.sglm_glm_epilogue_f64(p, 64, 8, 100, p, 1, p, None, 0, p, p, p, None, power, 1, p, p, 1 << 30,
                                         None) == -6, power
    assert ws > 0


def test_tweedie_estimator_family_validation():
    X, y = np.ones((4, 2)), np.ones(4)
    for kw in (dict(power=0.5), dict(power=0.0), dict(power=-1.0), dict(power=2.0, link="identity"),
               dict(power=1.0, link="identity")):
        with pytest.raises(NotImplementedError):
            sglm.TweedieRegressor(**kw).fit(X, y)
    with pytest.raises(NotImplementedError):
        sglm.GLM("Tweedie", power=0.5, alpha=0.1).fit(X, y)
    g = sglm.GLM("Gamma", alpha=0.1)
    assert g.model.power == 2 and g.model.kind == "tweedie" and g.model._link == 1
    assert sglm.GLM("Tweedie", power=1.5).model.kind == "tweedie"
    assert sglm.GLM("Poisson").model.kind == "poisson"
