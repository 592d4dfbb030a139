"""TweedieElasticNet without a GPU: the GLM dispatch of 'Poisson' / 'Gamma' / 'Tweedie' parameter sets that carry an
l1_ratio, the estimator's argument checks, the argument checks of sglm_pb_step_enet_f64 (every call below fails them
before any CUDA call), and the CPU reference of the penalised optimum (tests/tweedie_enet_reference.py) checked
against its KKT conditions and, at l1_ratio = 0, against the ridge reference."""
import ctypes

import numpy as np
import pytest

import _sglm_native as nat
import sglm
from _estimators import TweedieElasticNet, TweedieRegressor
import tweedie_enet_reference as eref
import tweedie_reference as tref

E_INVALID, E_SHAPE, E_ALIGN, E_WORKSPACE, E_UNSUPPORTED = -1, -2, -3, -4, -6


def test_dispatch_builds_elastic_net_for_l1_sets():
    g = sglm.GLM('Poisson', alpha=.1, l1_ratio=.5)
    assert type(g.model) is TweedieElasticNet and g.model.power == 1 and g.model.l1_ratio == .5
    assert g.model.kind == "tweedie_enet"
    g = sglm.GLM('Tweedie', power=1.5, alpha=.1, l1_ratio=1.0)
    assert type(g.model) is TweedieElasticNet and g.model.power == 1.5
    g = sglm.GLM('Gamma', alpha=.2, l1_ratio=.9, fit_intercept=False, max_iter=50, tol=1e-6)
    assert type(g.model) is TweedieElasticNet and g.model.power == 2
    assert g.model.get_params() == dict(power=2, alpha=.2, l1_ratio=.9, fit_intercept=False, link="auto",
                                        max_iter=50, tol=1e-6, warm_start=False)


def test_dispatch_zero_l1_ratio_or_alpha_builds_tweedie_regressor():
    g = sglm.GLM('Gamma', alpha=.1, l1_ratio=0)
    assert type(g.model) is TweedieRegressor and 'l1_ratio' not in g.kwargs and g.model.power == 2
    g = sglm.GLM('Poisson', alpha=0, l1_ratio=.5)
    assert type(g.model) is TweedieRegressor and 'l1_ratio' not in g.kwargs and g.model.power == 1
    g = sglm.GLM('Tweedie', power=1.5, alpha=.1)
    assert type(g.model) is TweedieRegressor and g.model.kind == "tweedie"


@pytest.mark.parametrize("kw", [dict(l1_ratio=1.5, alpha=.1), dict(l1_ratio=-.1, alpha=.1),
                                dict(l1_ratio=.5, alpha=-1.0), dict(l1_ratio=float("nan"), alpha=.1)])
def test_bad_l1_ratio_or_alpha_raise_value_error(kw):
    with pytest.raises(ValueError):
        sglm.GLM('Poisson', **kw)
    est = TweedieElasticNet(power=1, alpha=.1, l1_ratio=.5)
    est.set_params(**kw)
    with pytest.raises(ValueError):
        est.fit(np.ones((4, 2)), np.ones(4))


@pytest.mark.parametrize("kw", [dict(power=0.0), dict(power=0.5), dict(power=-1.0), dict(power=1.5, link="identity")])
def test_bad_power_or_link_raise_not_implemented(kw):
    with pytest.raises(NotImplementedError):
        sglm.GLM('Tweedie', alpha=.1, l1_ratio=.5, **kw)
    with pytest.raises(NotImplementedError):
        sglm.GLM('Poisson', alpha=.1, l1_ratio=.5, link="identity")


def test_unknown_keyword_raises_type_error():
    with pytest.raises(TypeError):
        sglm.GLM('Poisson', alpha=.1, l1_ratio=.5, reg_lambda=1.0)
    with pytest.raises(TypeError):
        sglm.GLM('Gamma', alpha=.1, l1_ratio=.5, solver="lbfgs")


def _state(C=8, B=4, ldw=8, ldq=8, ldb=64):
    """A PbState image with non-null fake device pointers (never dereferenced: the calls fail their checks)."""
    n = nat.lib().sglm_pb_state_words()
    words = np.full(n, 64, dtype=np.uint64)
    words[-4:] = [ldw, ldq, ldb, C | (B << 32)]
    return words


def test_pb_step_enet_argument_checks():
    lib = nat.lib()
    p = ctypes.c_void_p(64)
    odd = ctypes.c_void_p(72)
    big = 1 << 40
    st = _state()
    sp = st.ctypes.data_as(ctypes.c_void_p)
    assert lib.sglm_pb_enet_workspace_bytes(8, 8, 3) == 3 * (2 * 8 + 8) * 8
    assert lib.sglm_pb_enet_workspace_bytes(0, 8, 3) == 0
    assert lib.sglm_pb_step_enet_f64(None, p, p, p, 1, p, big, p, None) == E_INVALID
    assert b"null pointer" in lib.sglm_last_error()
    assert lib.sglm_pb_step_enet_f64(sp, None, p, p, 1, p, big, p, None) == E_INVALID
    assert lib.sglm_pb_step_enet_f64(sp, p, p, p, 0, p, big, p, None) == E_SHAPE          # no elastic-net model
    assert lib.sglm_pb_step_enet_f64(sp, p, p, p, 5, p, big, p, None) == E_SHAPE          # more than B = 4
    assert lib.sglm_pb_step_enet_f64(sp, p, p, None, 2, p, big, p, None) == E_INVALID
    assert lib.sglm_pb_step_enet_f64(sp, p, None, p, 2, p, big, p, None) == E_INVALID         # l1_ratio
    assert lib.sglm_pb_step_enet_f64(sp, p, p, p, 2, None, big, p, None) == E_INVALID
    assert lib.sglm_pb_step_enet_f64(sp, p, p, p, 2, p, big, None, None) == E_INVALID
    assert lib.sglm_pb_step_enet_f64(sp, p, p, p, 2, odd, big, p, None) == E_ALIGN
    need = lib.sglm_pb_enet_workspace_bytes(8, 8, 2)
    assert lib.sglm_pb_step_enet_f64(sp, p, p, p, 2, p, need - 8, p, None) == E_WORKSPACE
    bad = _state(ldw=4)                                                                   # ldw < C
    assert lib.sglm_pb_step_enet_f64(bad.ctypes.data_as(ctypes.c_void_p), p, p, p, 2, p, big, p, None) == E_SHAPE
    wide = _state(C=20000, ldw=20000, ldq=20000)             # the inner solve's shared memory (> 227 KB per model)
    assert lib.sglm_pb_step_enet_f64(wide.ctypes.data_as(ctypes.c_void_p), p, p, p, 2, p, big, p, None) == E_UNSUPPORTED


def _problem(n, p, seed, power):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((n, p))
    X[:, 1] = X[:, 0] + 0.3 * rng.standard_normal(n)            # correlated columns
    beta = np.zeros(p)
    beta[:3] = [0.4, -0.3, 0.2]
    mu = np.exp(X @ beta * 0.5 - 0.5)
    if power == 1:
        y = rng.poisson(mu).astype(np.float64)
    else:
        import synth_data
        y = synth_data.tweedie_draw(mu, seed, power)
    return X, y


@pytest.mark.parametrize("power", [1.0, 1.5, 2.0, 3.0])
@pytest.mark.parametrize("l1_ratio", [0.1, 0.5, 1.0])
@pytest.mark.parametrize("fit_intercept", [True, False])
def test_reference_satisfies_kkt(power, l1_ratio, fit_intercept):
    X, y = _problem(400, 8, 3, power)
    alpha = 0.2 * eref.alpha_max(X, y, l1_ratio, power, fit_intercept)
    w, b, f = eref.enet_fit(X, y, alpha, l1_ratio, fit_intercept, power)
    on, off, gb, _ = eref.kkt_residuals(X, y, w, b, alpha, l1_ratio, power, fit_intercept)
    assert on <= 1e-10 and off <= 1e-10 and gb <= 1e-10, (on, off, gb)
    assert 0 < np.count_nonzero(w) < len(w)                      # a sparse optimum: the L1 term is active
    assert f == pytest.approx(eref.objective(X, y, w, b, alpha, l1_ratio, power), rel=1e-15)


@pytest.mark.parametrize("power", [1.0, 1.5, 2.0, 3.0])
def test_reference_at_zero_l1_ratio_matches_ridge_reference(power):
    X, y = _problem(400, 8, 5, power)
    for fit_intercept in (True, False):
        w, b, _ = eref.enet_fit(X, y, 0.05, 0.0, fit_intercept, power)
        w_r, b_r, _ = tref.tweedie_fit(X, y, 0.05, fit_intercept, power)
        assert np.max(np.abs(w - w_r)) <= 1e-9 * max(1.0, np.max(np.abs(w_r)))
        assert abs(b - b_r) <= 1e-9 * max(1.0, abs(b_r))


def test_reference_null_model_above_alpha_max():
    X, y = _problem(400, 8, 7, 1.0)
    a = eref.alpha_max(X, y, 0.5, 1.0)
    w, b, _ = eref.enet_fit(X, y, 1.000001 * a, 0.5, True, 1.0)
    assert np.all(w == 0.0) and b == pytest.approx(np.log(y.mean()), rel=1e-12)
