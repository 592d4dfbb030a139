"""
Estimator objects behind `GLM.model` — the GPU counterparts of the scikit-learn classes
the reference instantiates (backend/sglm.py:2, :95-130): LinearRegression, Ridge, Lasso,
ElasticNet, TweedieRegressor (power 1 = Poisson, 2 = Gamma, any power > 1; log link), plus TweedieElasticNet
(the same families with an L1 + L2 penalty; no scikit-learn counterpart).  Same constructor keywords (unknown keywords raise
TypeError exactly as scikit-learn does, which is how stale kwargs such as `reg_lambda`
fail in the reference), same fitted attributes (`coef_`, `intercept_`, `n_iter_`,
`dual_gap_`), same `fit / predict / score`.  All arithmetic runs in libsglm_b200.so.
"""
import warnings

import numpy as np

import _engine as eng


class ConvergenceWarning(UserWarning):
    """Mirror of sklearn.exceptions.ConvergenceWarning (a warning, not an error)."""


class _Base:
    kind = None
    _link = 0

    def get_params(self, deep=True):
        import inspect
        return {k: getattr(self, k) for k in inspect.signature(type(self).__init__).parameters if k != "self"}

    def set_params(self, **params):
        for k, v in params.items():
            if k not in self.get_params():
                raise ValueError(f"Invalid parameter {k!r} for estimator {type(self).__name__}")
            setattr(self, k, v)
        return self

    def __repr__(self):
        import inspect
        sig = inspect.signature(type(self).__init__).parameters
        diff = [f"{k}={getattr(self, k)!r}" for k, p in sig.items()
                if k != "self" and getattr(self, k) != p.default]
        return f"{type(self).__name__}({', '.join(diff)})"

    # -- shared fit path: statistics -> centred problem -> solver -> intercept
    def _check_supported(self):
        if getattr(self, "positive", False):
            raise NotImplementedError("positive=True is not part of the sGLM hot path")
        if getattr(self, "selection", "cyclic") != "cyclic":
            raise NotImplementedError("selection='random' is not part of the sGLM hot path")

    def _spec(self, problem):
        raise NotImplementedError

    def fit(self, X, y, sample_weight=None):
        if sample_weight is not None:
            raise NotImplementedError("sample_weight is never passed by the reference (backend/sglm.py:241)")
        self._check_supported()
        Xd = eng.device_matrix(X)
        yd = eng.device_vector(y)
        if Xd.shape[0] != yd.shape[0]:
            raise ValueError(f"Found input variables with inconsistent numbers of samples: "
                             f"[{Xd.shape[0]}, {yd.shape[0]}]")
        if Xd.shape[0] < 1:
            raise ValueError("Found array with 0 sample(s) while a minimum of 1 is required.")
        C = Xd.shape[1]
        G = eng.suffstats(Xd, yd[:, None])
        _require_finite(G)
        prob = eng.center(G[0], None, C, 1, 0, self.fit_intercept)
        eng.fetch_scalars([prob])
        spec = self._spec(prob)
        W, info, status = eng.solve_models([spec], C)
        b, _ = eng.finalize(W, C, 1, [spec])
        self.coef_ = W[0, :C].cpu().numpy()
        self.intercept_ = float(b[0].item()) if self.fit_intercept else 0.0
        self.n_features_in_ = C
        self._after_fit(info[0], int(status[0]))
        if not (np.isfinite(self.coef_).all() and np.isfinite(self.intercept_)):
            if status[0] == 2:
                raise np.linalg.LinAlgError("Matrix is singular: X'X + alpha*I is not positive definite")
            raise ValueError("Coordinate descent iterations resulted in non-finite parameter values. The input "
                             "data may contain large values and need to be preprocessed.")
        return self

    def _after_fit(self, info, status):
        pass

    def predict(self, X):
        Xd = eng.device_matrix(X)
        out = eng.predict(Xd, self.coef_, self.intercept_, self._link)
        return out if eng.is_torch(eng._values(X)) else out.cpu().numpy()

    def score(self, X, y, sample_weight=None):
        Xd, yd = eng.device_matrix(X), eng.device_vector(y)
        s, _ = eng.score_sums(Xd, yd, self.coef_, self.intercept_, self._link)
        return eng.r2_from_sums(s)


def _require_finite(G):
    import torch
    if not bool(torch.isfinite(G).all().item()):
        raise ValueError("Input contains NaN, infinity or a value too large for dtype('float64').")


class LinearRegression(_Base):
    """OLS (reference: backend/sglm.py:96-101; sklearn _base.py:700-756)."""
    kind = "ols"

    def __init__(self, *, fit_intercept=True, copy_X=True, tol=1e-6, n_jobs=None, positive=False):
        self.fit_intercept, self.copy_X, self.tol, self.n_jobs, self.positive = \
            fit_intercept, copy_X, tol, n_jobs, positive

    def _spec(self, problem):
        return eng.ModelSpec(problem, "ols", tol=self.tol)      # tol = lstsq cond (_base.py:750-753)


class Ridge(_Base):
    """Ridge, alpha NOT scaled by n (reference: backend/sglm.py:102-105; sklearn _ridge.py:215-227)."""
    kind = "ridge"

    def __init__(self, alpha=1.0, *, fit_intercept=True, copy_X=True, max_iter=None, tol=1e-4,
                 solver="auto", positive=False, random_state=None):
        self.alpha, self.fit_intercept, self.copy_X, self.max_iter, self.tol = \
            alpha, fit_intercept, copy_X, max_iter, tol
        self.solver, self.positive, self.random_state = solver, positive, random_state

    def _spec(self, problem):
        if self.solver not in ("auto", "cholesky"):
            raise NotImplementedError(f"Ridge solver={self.solver!r}: only the reference's default (cholesky) is built")
        if self.alpha < 0:
            raise ValueError("The 'alpha' parameter of Ridge must be a float in the range [0.0, inf).")
        return eng.ModelSpec(problem, "ridge", alpha=self.alpha)


class ElasticNet(_Base):
    """ElasticNet by cyclic coordinate descent (reference: backend/sglm.py:109-110;
    sklearn _coordinate_descent.py:1095-1281, _cd_fast.pyx:243-506)."""
    kind = "enet"

    def __init__(self, alpha=1.0, *, l1_ratio=0.5, fit_intercept=True, precompute=False, max_iter=1000,
                 copy_X=True, tol=1e-4, warm_start=False, positive=False, random_state=None,
                 selection="cyclic"):
        self.alpha, self.l1_ratio, self.fit_intercept, self.precompute = alpha, l1_ratio, fit_intercept, precompute
        self.max_iter, self.copy_X, self.tol, self.warm_start = max_iter, copy_X, tol, warm_start
        self.positive, self.random_state, self.selection = positive, random_state, selection

    def _spec(self, problem):
        init = getattr(self, "coef_", None) if self.warm_start else None
        if self.alpha == 0:
            warnings.warn("With alpha=0, this algorithm does not converge well. You are advised to use the "
                          "LinearRegression estimator", stacklevel=3)
        return eng.ModelSpec(problem, "enet", alpha=self.alpha, l1_ratio=self.l1_ratio, max_iter=self.max_iter,
                             tol=self.tol, coef_init=init)

    def _after_fit(self, info, status):
        self.dual_gap_ = float(info[0])
        self.n_iter_ = int(info[2])
        if status == 1:
            warnings.warn(f"Objective did not converge. You might want to increase the number of iterations, "
                          f"check the scale of the features or consider increasing regularisation. "
                          f"Duality gap: {info[0]:.6e}, tolerance: {info[1]:.3e}", ConvergenceWarning, stacklevel=3)


class Lasso(ElasticNet):
    """Lasso = ElasticNet(l1_ratio=1) (reference: backend/sglm.py:106-108)."""
    kind = "lasso"

    def __init__(self, alpha=1.0, *, fit_intercept=True, precompute=False, copy_X=True, max_iter=1000,
                 tol=1e-4, warm_start=False, positive=False, random_state=None, selection="cyclic"):
        super().__init__(alpha=alpha, l1_ratio=1.0, fit_intercept=fit_intercept, precompute=precompute,
                         copy_X=copy_X, max_iter=max_iter, tol=tol, warm_start=warm_start, positive=positive,
                         random_state=random_state, selection=selection)

    def get_params(self, deep=True):
        p = super().get_params(deep)
        p.pop("l1_ratio", None)
        return p


class TweedieRegressor(_Base):
    """Tweedie GLM with log link (reference: backend/sglm.py:112-117 builds TweedieRegressor(power=1)
    for 'Poisson', power=2 for 'Gamma', TweedieRegressor(**kwargs) for 'Tweedie'; sklearn
    _glm/glm.py:185-339).  Fitted on the GPU to the optimum of  mean(l(y, eta)) + alpha/2 |w|^2
    with sklearn's HalfTweedieLoss l — power 1 by IRLS/Newton, power > 1 by the batched solver
    with one model; `score` is the family's D^2.  Power <= 0, 0 < power < 1 and the identity
    link are not built."""
    _link = 1

    @property
    def kind(self):
        return "poisson" if self.power == 1 else "tweedie"

    def __init__(self, *, power=0.0, alpha=1.0, fit_intercept=True, link="auto", solver="lbfgs",
                 max_iter=100, tol=1e-4, warm_start=False, verbose=0):
        self.power, self.alpha, self.fit_intercept, self.link = power, alpha, fit_intercept, link
        self.solver, self.max_iter, self.tol, self.warm_start, self.verbose = solver, max_iter, tol, warm_start, verbose

    def _check_family(self):
        if not (self.power == 1 or self.power > 1) or self.link not in ("auto", "log"):
            raise NotImplementedError("the GPU path builds the Tweedie families with log link and power 1 (Poisson) "
                                      "or power > 1 (Gamma, compound Poisson-Gamma, inverse Gaussian, ...); "
                                      f"power={self.power!r}, link={self.link!r} is not built")

    def _check_y(self, yd):
        """scikit-learn's range check of HalfTweedieLoss: y >= 0 for power < 2, y > 0 for power >= 2."""
        lo = float(yd.min().item()) if yd.numel() else 0.0
        if not (lo >= 0) or (self.power >= 2 and not (lo > 0)):
            raise ValueError(f"Some value(s) of y are out of the valid range of the loss '{eng._loss_name(self.power)}'.")

    def fit(self, X, y, sample_weight=None):
        if sample_weight is not None:
            raise NotImplementedError("sample_weight is never passed by the reference")
        self._check_family()
        Xd, yd = eng.device_matrix(X), eng.device_vector(y)
        import torch
        if self.power == 1:
            if bool((yd < 0).any().item()):
                raise ValueError("Some value(s) of y are out of the valid range of the loss 'HalfPoissonLoss'.")
        else:
            self._check_y(yd)
        if not bool(torch.isfinite(Xd).all().item()):
            raise ValueError("Input X contains NaN or infinity.")
        ci = getattr(self, "coef_", None) if self.warm_start else None
        ii = getattr(self, "intercept_", None) if self.warm_start else None
        if self.power == 1:
            self.coef_, self.intercept_, self.n_iter_ = eng.poisson_irls(
                Xd, yd, self.alpha, self.fit_intercept, None, self.max_iter, self.tol, ci, ii)
        else:
            m = eng.PoissonModel(self.alpha, self.fit_intercept, max_iter=self.max_iter, tol=self.tol, coef_init=ci,
                                 intercept_init=ii)
            W, b, n_it, _ = eng.tweedie_grid_batched(Xd, yd[:, None], [m], None, self.power)
            self.coef_ = W[0].cpu().numpy()
            self.intercept_ = float(b[0].item()) if self.fit_intercept else 0.0
            self.n_iter_ = int(n_it[0])
        self.n_features_in_ = Xd.shape[1]
        return self

    def score(self, X, y, sample_weight=None):
        self._check_family()
        Xd, yd = eng.device_matrix(X), eng.device_vector(y)
        if self.power == 1:
            s, _ = eng.score_sums(Xd, yd, self.coef_, self.intercept_, 1)
            return eng.poisson_d2_from_sums(s)
        self._check_y(yd)
        s, _ = eng.score_sums(Xd, yd, self.coef_, self.intercept_, power=self.power)
        return eng.tweedie_d2_from_sums(s, self.power)


class TweedieElasticNet(_Base):
    """Tweedie GLM with log link and an elastic-net penalty — an extension with no scikit-learn counterpart:

        argmin  mean(l(y, eta)) + alpha l1_ratio |w|_1 + alpha (1 - l1_ratio)/2 |w|^2,   eta = X w + b (b unpenalised)

    with sklearn's HalfTweedieLoss l of `power` (1 = Poisson, 2 = Gamma, any power > 1), the L1 term scaled by the
    mean loss as in glmnet / pyglmnet and this project's ElasticNet.  At l1_ratio = 0 this is TweedieRegressor's
    objective.  Fitted by the batched solver with one model for every power (proximal-Newton steps: the quadratic
    model of the chord step solved by Gram coordinate descent); `score` is the family's D^2."""
    _link = 1
    kind = "tweedie_enet"

    def __init__(self, *, power=0.0, alpha=1.0, l1_ratio=0.5, fit_intercept=True, link="auto", max_iter=100,
                 tol=1e-4, warm_start=False):
        self.power, self.alpha, self.l1_ratio, self.fit_intercept, self.link = power, alpha, l1_ratio, fit_intercept, link
        self.max_iter, self.tol, self.warm_start = max_iter, tol, warm_start
        self._check_params()
        self._check_family()

    _check_family = TweedieRegressor._check_family
    _check_y = TweedieRegressor._check_y
    score = TweedieRegressor.score

    def _check_params(self):
        if not (0.0 <= self.l1_ratio <= 1.0):
            raise ValueError(f"The 'l1_ratio' parameter of TweedieElasticNet must be a float in the range [0.0, 1.0]; "
                             f"got {self.l1_ratio!r}.")
        if not (self.alpha >= 0.0):
            raise ValueError(f"The 'alpha' parameter of TweedieElasticNet must be a float in the range [0.0, inf); "
                             f"got {self.alpha!r}.")

    def fit(self, X, y, sample_weight=None):
        if sample_weight is not None:
            raise NotImplementedError("sample_weight is never passed by the reference")
        self._check_params()
        self._check_family()
        Xd, yd = eng.device_matrix(X), eng.device_vector(y)
        import torch
        self._check_y(yd)
        if not bool(torch.isfinite(Xd).all().item()):
            raise ValueError("Input X contains NaN or infinity.")
        ci = getattr(self, "coef_", None) if self.warm_start else None
        ii = getattr(self, "intercept_", None) if self.warm_start else None
        m = eng.PoissonModel(self.alpha, self.fit_intercept, max_iter=self.max_iter, tol=self.tol, coef_init=ci,
                             intercept_init=ii, l1_ratio=self.l1_ratio)
        W, b, n_it, _ = eng.tweedie_grid_batched(Xd, yd[:, None], [m], None, float(self.power))
        self.coef_ = W[0].cpu().numpy()
        self.intercept_ = float(b[0].item()) if self.fit_intercept else 0.0
        self.n_iter_ = int(n_it[0])
        self.n_features_in_ = Xd.shape[1]
        return self
