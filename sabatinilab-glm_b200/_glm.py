"""
sglm — drop-in for the reference module `backend/sglm.py` (identical to `backend/sglm_.py`):
the `GLM` wrapper and `calc_R2`, with every fit / prediction / score executed by the
B200 kernels of libsglm_b200.so instead of scikit-learn on the host.

Mirrors (reference file:line): constructor dispatch backend/sglm.py:59-147, `fit` :225-251,
`fit_set` :254-312, `get_residuals` :314-331, `predict` :333-347, `neg_mse_score` :150-167,
`r2_score` :169-184, `pca_fit` :186-223, `log_likelihood` :349-385, `calc_R2` :388-408.

Deliberate deviations (crash / hang fixes, documented in DESIGN.md):
  * Poisson: the reference fits and then raises AttributeError because it reads the
    pyglmnet attributes `beta_/beta0_` (backend/sglm.py:246-250); here `coef_/intercept_`
    are mapped, so Poisson fits are usable.
  * Gamma / Tweedie: the GPU path fits power 1 and any power > 1 with log link; power <= 0,
    0 < power < 1 and link='identity' raise NotImplementedError.  With all-zero y and
    1 < power < 2 the fit raises ValueError (scikit-learn returns an intercept of -inf).
  * Poisson / Gamma / Tweedie with `l1_ratio` (an extension: the reference's TweedieRegressor has no
    such keyword and raises TypeError): with l1_ratio and alpha both non-zero the model is a
    TweedieElasticNet, mean loss + alpha (l1_ratio |w|_1 + (1 - l1_ratio)/2 |w|^2) as in pyglmnet,
    which the reference's users fitted before; l1_ratio == 0 or alpha == 0 drops the keyword and
    builds TweedieRegressor, as l1_ratio == 0 builds Ridge for the Gaussian family.
  * Logistic / Multinomial are outside the hot-path scope (SURVEY.md §8) and raise
    NotImplementedError.
"""
import time

import numpy as np

import _engine as eng
from _estimators import (ConvergenceWarning, ElasticNet, Lasso, LinearRegression, Ridge,  # noqa: F401
                         TweedieElasticNet, TweedieRegressor)


class NotYetImplementedError(NameError, NotImplementedError):
    """The reference raises an undefined name here (backend/sglm.py:124-126), i.e. a
    NameError; this class is caught by both `except NameError` and NotImplementedError."""


_GAUSSIAN_NAMES = {"Logistic", "Multinomial", "Gaussian", "Normal", "PCA Gaussian", "PCA Normal"}


class GLM():
    """Generalized Linear Model wrapper with the reference's interface; `self.model` is a
    GPU estimator (see _estimators.py) exposing the scikit-learn attribute names."""

    model = None
    model_name_options = {'Normal', 'Gaussian', 'Poisson', 'Tweedie', 'Gamma', 'Logistic', 'Binomial', 'Multinomial'}
    tweedie_lookup = {'Normal': 0, 'Gaussian': 0, 'Poisson': 1, 'Gamma': 2}

    def __init__(self, model_name, beta0_=None, beta_=None, score_method='mse', *args, **kwargs):
        if 'warm_start' not in kwargs and (beta0_ is not None or isinstance(beta_, np.ndarray)):
            kwargs['warm_start'] = True

        self.model_name = model_name
        # second-generation attributes (sglm/sglm/models/sglm.py:69-71): `closed_form` is switched
        # on by the caller after construction and turns `fit` into an un-penalised least-squares fit
        self.closed_form = False
        if 'fit_intercept' in kwargs:
            self.fit_intercept = kwargs['fit_intercept']
        if model_name in {'Normal', 'Gaussian'}:
            # estimator choice by (alpha, l1_ratio) — backend/sglm.py:96-110
            if 'alpha' in kwargs and kwargs['alpha'] == 0:
                for key in ('alpha', 'l1_ratio', 'max_iter'):
                    kwargs.pop(key)                      # KeyError when absent, as in the reference
                kwargs.pop('warm_start', None)
                Base = LinearRegression
            elif 'l1_ratio' in kwargs and kwargs['l1_ratio'] == 0:
                del kwargs['l1_ratio']
                kwargs.pop('warm_start', None)
                Base = Ridge
            elif 'l1_ratio' in kwargs and kwargs['l1_ratio'] == 1:
                del kwargs['l1_ratio']
                Base = Lasso
            else:
                Base = ElasticNet
        elif model_name in {'Poisson', 'Gamma', 'Tweedie'}:
            if model_name != 'Tweedie':
                kwargs['power'] = self.tweedie_lookup[model_name]
            Base = TweedieRegressor
            if 'l1_ratio' in kwargs:
                if kwargs['l1_ratio'] == 0 or kwargs.get('alpha', 1.0) == 0:
                    del kwargs['l1_ratio']
                else:
                    Base = TweedieElasticNet
        elif model_name in {'Logistic', 'Multinomial'}:
            raise NotImplementedError("Logistic/Multinomial GLMs are outside the B200 hot-path scope")
        elif model_name in {'PCA Normal', 'PCA Gaussian'}:
            Base = LinearRegression
        else:
            print('Distribution not yet implemented.')
            raise NotYetImplementedError("name 'NotYetImplementedError' is not defined")

        self.Base = Base
        self.kwargs = kwargs
        self.model = self.Base(*args, **kwargs)

        if beta0_ is not None:
            self.model.intercept_ = beta0_
            self.beta0_ = beta0_
        if isinstance(beta_, np.ndarray):
            self.beta_ = np.copy(beta_)
            self.model.coef_ = self.beta_

        self.score = self.r2_score if score_method == 'r2' else self.neg_mse_score

    # ------------------------------------------------------------------ scores
    def neg_mse_score(self, X, y):
        """-mean((y - predict(X))^2) (backend/sglm.py:150-167) — one fused pass over X."""
        Xd, yd = eng.device_matrix(X), eng.device_vector(y)
        s, _ = eng.score_sums(Xd, yd, self.model.coef_, self.model.intercept_, self.model._link)
        return -float(s[1] / s[0])

    def r2_score(self, X, y):
        """model.score(X, y): R^2, or D^2 for the Poisson / Gamma / Tweedie families (backend/sglm.py:169-184)."""
        return self.model.score(X, y)

    # ------------------------------------------------------------------ fits
    def pca_fit(self, X, y):
        """backend/sglm.py:186-223 rotates X by a full-rank PCA, fits, and rotates the
        coefficients back — for a full set of components that is the un-rotated fit itself,
        so the GPU path fits directly (the CV driver discards this result anyway,
        backend/sglm_cv.py:275-282)."""
        if self.model_name in {'Normal', 'Gaussian'}:
            self.model.alpha = 0.1 if 'alpha' not in self.kwargs else self.kwargs['alpha']
            self.model.l1_ratio = 0.5 if 'l1_ratio' not in self.kwargs else self.kwargs['l1_ratio']
        self.pca = None
        self.fit(X, y)
        self.beta_ = np.asarray(self.coef_).reshape(-1)
        self.coef_ = self.beta_
        self.beta0_ = np.asarray(self.intercept_).reshape(-1)
        self.intercept_ = self.beta0_

    def fit(self, X, y, *args):
        if self.closed_form:
            # sglm/sglm/models/sglm.py:263-293: lstsq on [X | 1]; same least-squares solution as the
            # centred OLS solve of the GPU path (minimum-norm fallback when rank-deficient)
            ols = LinearRegression(fit_intercept=getattr(self, 'fit_intercept', True))
            ols.fit(X, y)
            self.coef_ = self.beta_ = ols.coef_
            self.intercept_ = self.beta0_ = ols.intercept_
            self.full_betas_ = np.concatenate([ols.coef_, [ols.intercept_]]) if ols.fit_intercept else ols.coef_
            self.model.coef_, self.model.intercept_ = self.coef_, self.intercept_
            return
        self.model.fit(X, y, *args)
        # attribute mapping of backend/sglm.py:246-251 (Poisson mapped too, see module docstring)
        self.coef_ = self.model.coef_
        self.beta_ = self.coef_
        self.intercept_ = self.model.intercept_
        self.beta0_ = self.intercept_

    def fit_set(self, X, y, X_test, y_test, cv_coefs,
                cv_intercepts, cv_scores_train, cv_scores_test,
                iter_cv, *args, resids=[], mean_resids=[], id_fit='None', verbose=0):
        """Fit and write the fold's results in place (backend/sglm.py:254-312)."""
        if verbose > 1:
            start = time.time()
            print(f'Fitting: {self.kwargs} — {id_fit}')
        self.fit(X, y, *args)
        if verbose > 1:
            print(f'Done with: {self.kwargs} — {id_fit} — in {time.time() - start}')
        cv_coefs[:, iter_cv] = self.coef_
        cv_intercepts[iter_cv] = self.intercept_
        cv_scores_train[iter_cv] = self.score(X, y)
        cv_scores_test[iter_cv] = self.score(X_test, y_test)
        residuals, mean_residuals = self.get_residuals(X_test, y_test)
        resids.append(residuals)
        mean_resids.append(mean_residuals)

    def get_residuals(self, X, y):
        """(y - predict(X), y - mean(y)) (backend/sglm.py:314-331)."""
        Xd, yd = eng.device_matrix(X), eng.device_vector(y)
        s, resid = eng.score_sums(Xd, yd, self.model.coef_, self.model.intercept_, self.model._link,
                                  want_resid=True)
        mean_resid = yd - (s[2] / s[0])
        if eng.is_torch(eng._values(X)):
            return resid, mean_resid
        return resid.cpu().numpy(), mean_resid.cpu().numpy()

    def predict(self, X):
        """model.predict(X) (backend/sglm.py:333-347)."""
        return self.model.predict(X)

    def log_likelihood(self, prediction, truth):
        """Gaussian log-likelihood of residuals (backend/sglm.py:349-385; other families
        are unimplemented in the reference as well)."""
        if self.model_name in {'Normal', 'Gaussian'}:
            resid = np.asarray(truth, dtype=np.float64) - np.asarray(prediction, dtype=np.float64)
            std = np.std(resid)
            return float(np.sum(-0.5 * np.log(2 * np.pi * std * std) - resid ** 2 / (2 * std * std)))
        raise NotYetImplementedError("name 'NotYetImplementedError' is not defined")


def fit_GLM(X, y, model_name='Gaussian', *args, **kwargs):
    """Second-generation convenience (sglm/sglm/models/sglm.py:345-364): build, fit, return."""
    glm = GLM(model_name, *args, **kwargs)
    glm.fit(X, y)
    return glm


def calc_R2(residuals, mean_residuals):
    """1 - RSS/TSS with TSS == 0 -> 0 (backend/sglm.py:388-408)."""
    rss = np.sum(np.asarray(residuals) ** 2)
    tss = np.sum(np.asarray(mean_residuals) ** 2)
    return 0 if tss == 0 else 1 - rss / tss
