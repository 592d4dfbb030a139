"""The other BASELINE.json configurations on one B200, each with the reference's CPU path timed beside it
(SURVEY.md §8d): configs[0] single ElasticNet fit 100k x 410, configs[1] Ridge CV 5 folds x 20 alphas 500k x 1220,
configs[3] Poisson alpha sweep 20 alphas x 5 folds (+ refits) 1M x 800, and the same sweep for the Gamma family (c4g)
and the Tweedie family with power 1.5 (c4t) on a response of that family, and the Poisson sweep with elastic-net
penalties (c4en: 20 alphas x l1_ratio 0.1 / 0.5 / 0.9 x (5 folds + refit) = 360 fits).  One JSON line per configuration:
device-resident time (CUDA events, warm-up excluded), end-to-end time from host numpy arrays, per-entry-point
milliseconds, and the CPU baseline (scikit-learn through the oracle port, bounded sample, extrapolated and labelled).

    python scripts/config_bench.py [c1] [c2] [c4] [c4g] [c4t] [c4en] [--no-cpu]     (default: c1 c2 c4)
"""
import json
import os
import sys
import time
import warnings

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "sabatinilab-glm_b200"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import synth_data  # noqa: E402
import _engine  # noqa: E402
import _sglm_native as nat  # noqa: E402
import sglm  # noqa: E402
import sglm_cv  # noqa: E402
import sglm_pp  # noqa: E402

warnings.filterwarnings("ignore")
CORES = len(os.sched_getaffinity(0))


def session(T, P, lo, hi, seed, poisson=False, power=None):
    shifts = [0] + [s for s in range(lo, hi + 1) if s != 0]
    X0_h = synth_data.synth_base(T, P, seed)
    X0 = torch.from_numpy(X0_h).cuda()
    beta = torch.from_numpy(synth_data.synth_kernels(P, shifts, seed)).cuda()
    h_lo, h_hi = max(0, hi), max(0, -lo)
    X = sglm_pp.timeshift_multiple(X0, shift_amt_list=shifts)[h_lo:T - h_hi]
    torch.manual_seed(seed)
    s = X @ beta
    if poisson:
        z = (s - s.mean()) / s.std()
        y = torch.poisson(torch.exp(0.3 * z - 1.0))
    elif power is not None:
        z = (s - s.mean()) / s.std()
        mu = torch.exp(0.3 * z - 1.0).cpu().numpy()
        y = torch.from_numpy(synth_data.tweedie_draw(mu, seed, power)).cuda()
    else:
        y = s + 1.5 * s.std() * torch.randn_like(s)
        y = (y - y.mean()) / y.std()
    n = X.shape[0]
    del X, s
    return X0_h, X0, shifts, (h_lo, T - h_hi), y.contiguous(), n


def timed(fn, reps=3, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    nat.enable_timing(True)
    nat.collect_timing()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        r = fn()
    e1.record()
    torch.cuda.synchronize()
    per = {k: v[1] / reps for k, v in nat.collect_timing().items()}
    nat.enable_timing(False)
    return e0.elapsed_time(e1) / reps / 1e3, r, per


def cpu_fit_seconds(make_estimator, X, y, reps=1):
    t0 = time.perf_counter()
    for _ in range(reps):
        make_estimator().fit(X, y)
    return (time.perf_counter() - t0) / reps


def host_design(X0_h, shifts, T_s):
    from oracle import sglm_oracle as orc
    Xd = orc.timeshift_multiple(X0_h[:T_s], shift_amt_list=shifts)
    return Xd[~np.isnan(Xd).any(axis=1)]


def run_c1(cpu):
    from sklearn.linear_model import ElasticNet
    X0_h, X0, shifts, (lo, hi), y, n = session(100_000, 10, -20, 20, 1)
    y_h = y.cpu().numpy()

    def dev():
        d = sglm_pp.timeshift_multiple(X0, shift_amt_list=shifts)[lo:hi]
        g = sglm.GLM("Gaussian", alpha=0.01, l1_ratio=0.5)
        g.fit(d, y)
        return g

    def e2e():
        d = sglm_pp.timeshift_multiple(X0_h, shift_amt_list=shifts, device=True).dropna()
        g = sglm.GLM("Gaussian", alpha=0.01, l1_ratio=0.5)
        g.fit(d, y_h)
        return g
    sec, _, per = timed(dev)
    sec_e, g, _ = timed(e2e)
    line = {"config": "c1 (BASELINE configs[0]): single Gaussian ElasticNet fit (alpha 0.01, l1_ratio 0.5), 100k timepoints x "
                      "10 predictors x 41 shifts = 410 columns, lag gather included", "fits": 1, "seconds": sec,
            "fits_per_s": 1 / sec, "e2e_seconds_numpy_in": sec_e, "n_iter": int(g.model.n_iter_), "per_entry_ms": per}
    if cpu:
        t0 = time.perf_counter()
        Xd = host_design(X0_h, shifts, 100_000)
        t_gather = time.perf_counter() - t0
        t_fit = cpu_fit_seconds(lambda: ElasticNet(alpha=0.01, l1_ratio=0.5), Xd, y_h)
        ref = ElasticNet(alpha=0.01, l1_ratio=0.5).fit(Xd, y_h)
        line["cpu_baseline"] = {"seconds": t_gather + t_fit, "fits_per_s": 1 / (t_gather + t_fit), "cores": CORES, "kind": "port",
                                "sample": "the full configuration (host lag gather %.2f s + sklearn ElasticNet.fit %.2f s)" % (t_gather, t_fit),
                                "coef_rel_err_gpu_vs_cpu": float(np.max(np.abs(g.coef_ - ref.coef_)) / np.max(np.abs(ref.coef_))),
                                "n_iter_cpu": int(ref.n_iter_)}
    return line


def run_c2(cpu):
    from sklearn.linear_model import Ridge
    X0_h, X0, shifts, (lo, hi), y, n = session(500_000, 20, -30, 30, 2)
    folds_h = synth_data.synth_folds(n, 5, 2)
    folds = [(torch.from_numpy(a).cuda(), torch.from_numpy(b).cuda()) for a, b in folds_h]
    y_h = y.cpu().numpy()
    grid = [dict(alpha=float(a), l1_ratio=0, max_iter=1000, fit_intercept=True) for a in np.logspace(-3, 3, 20)]

    def dev():
        d = sglm_pp.timeshift_multiple(X0, shift_amt_list=shifts)[lo:hi]
        return sglm_cv.cv_glm_mult_params(d, y, folds, "Gaussian", [dict(g) for g in grid], score_method="r2")

    def e2e():
        d = sglm_pp.timeshift_multiple(X0_h, shift_amt_list=shifts, device=True).dropna()
        return sglm_cv.cv_glm_mult_params(d, y_h, folds_h, "Gaussian", [dict(g) for g in grid], score_method="r2")
    sec, r, per = timed(dev)
    sec_e, _, _ = timed(e2e, reps=2, warm=1)
    line = {"config": "c2 (BASELINE configs[1]): Ridge CV grid 5 folds x 20 alphas (+ refits = 120 fits), 500k timepoints x "
                      "20 predictors x 61 shifts = 1220 columns, lag gather included", "fits": 120, "seconds": sec,
            "fits_per_s": 120 / sec, "e2e_seconds_numpy_in": sec_e, "e2e_fits_per_s": 120 / sec_e,
            "best_params": r["best_params"], "per_entry_ms": per}
    if cpu:
        Ts = 50_000
        Xd = host_design(X0_h, shifts, Ts)
        ys = y_h[:Xd.shape[0]]
        t_fit = cpu_fit_seconds(lambda: Ridge(alpha=1.0), Xd, ys, reps=2)
        per_fit_full = t_fit * (n * 0.8 / Xd.shape[0])
        line["cpu_baseline"] = {"fits_per_s": 1 / per_fit_full * 2.0, "cores": CORES, "kind": "port", "extrapolated": True,
                                "sample": "sklearn Ridge.fit (cholesky: X'X per fit) on %d x 1220: %.2f s per fit; extrapolated linearly in "
                                          "the rows to a 400k-row fold fit (%.1f s) and to the reference's 4 fold threads (6 fits in 3 "
                                          "rounds = x2.0)" % (Xd.shape[0], t_fit, per_fit_full)}
    return line


def run_c4(cpu):
    from sklearn.linear_model import TweedieRegressor
    X0_h, X0, shifts, (lo, hi), y, n = session(1_000_000, 20, -20, 19, 4, poisson=True)
    folds_h = synth_data.synth_folds(n, 5, 4)
    folds = [(torch.from_numpy(a).cuda(), torch.from_numpy(b).cuda()) for a, b in folds_h]
    y_h = y.cpu().numpy()
    grid = [dict(alpha=float(a), model_name="Poisson") for a in np.logspace(-4, 1, 20)]      # backend/sglm_cv.py:288
    d_keep = sglm_pp.timeshift_multiple(X0, shift_amt_list=shifts)[lo:hi]

    def dev():
        d = sglm_pp.timeshift_multiple(X0, shift_amt_list=shifts)[lo:hi]
        return sglm_cv.cv_glm_mult_params(d, y, folds, "Poisson", [dict(g) for g in grid], score_method="r2")
    sec, r, per = timed(dev, reps=2, warm=1)
    diag = _engine.last_poisson_batch
    line = {"config": "c4 (BASELINE configs[3]): Poisson GLM (log link, L2) alpha sweep logspace(-4, 1, 20) x (5 folds + refit) = 120 "
                      "fits, 1M timepoints x 20 predictors x 40 shifts = 800 columns, every fit driven to its optimum (step bound 1e-8)",
            "fits": 120, "seconds": sec, "fits_per_s": 120 / sec, "best_params": r["best_params"], "batch": diag,
            "n_iter_min_max": [int(min(np.min(x["_fit_info"]["n_iter"]) for x in r["full_cv_results"])),
                               int(max(np.max(x["_fit_info"]["n_iter"]) for x in r["full_cv_results"]))],
            "per_entry_ms": per}
    # algorithmic work of one batched iteration: two fp64 GEMMs of 2 T C B flops, 16 T B bytes of epilogue traffic
    if "sglm_pb_eta_f64" in per and diag:
        rounds = diag[0]["rounds"]
        B = 128
        line["roofline_pb_gemm"] = {"bound": "fp64 pipe", "eta_TFLOPs": 2.0 * n * 800 * B * rounds / (per["sglm_pb_eta_f64"] / 1e3) / 1e12,
                                    "xt_r_TFLOPs": 2.0 * n * 800 * B * rounds / (per["sglm_pb_xt_r_f64"] / 1e3) / 1e12,
                                    "note": "issued flops incl. the 8 padding columns (B = 120 models padded to 128); nominal FP64 ~40 TFLOP/s"}
    if cpu:
        Ts = 60_000
        Xd = host_design(X0_h, shifts, Ts)
        ys = y_h[:Xd.shape[0]]
        secs = []
        for a in (1e-4, 1e-1, 10.0):
            secs.append(cpu_fit_seconds(lambda: TweedieRegressor(power=1, alpha=a, max_iter=100), Xd, ys))
        per_fit = float(np.mean(secs)) * (n * 0.8 / Xd.shape[0])
        line["cpu_baseline"] = {"fits_per_s": 1 / per_fit * 2.0, "cores": CORES, "kind": "port", "extrapolated": True,
                                "sample": "TweedieRegressor(power=1, max_iter=100, default lbfgs, tol 1e-4) at alpha 1e-4 / 1e-1 / 10 on "
                                          "%d x 800: %s s; extrapolated linearly in the rows to an 800k-row fold fit (%.1f s per fit) and "
                                          "to the reference's 4 fold threads (x2.0).  The reference wrapper itself raises after the fit "
                                          "(backend/sglm.py:246-250)" % (Xd.shape[0], [round(s, 2) for s in secs], per_fit)}
    del d_keep
    return line


def run_c4_family(name, model_name, power):
    """c4 with the response and the family of `model_name` (log link): the same design, folds and alpha sweep."""
    X0_h, X0, shifts, (lo, hi), y, n = session(1_000_000, 20, -20, 19, 4, power=power)
    folds_h = synth_data.synth_folds(n, 5, 4)
    folds = [(torch.from_numpy(a).cuda(), torch.from_numpy(b).cuda()) for a, b in folds_h]
    extra = {} if model_name == "Gamma" else {"power": power}
    grid = [dict(alpha=float(a), model_name=model_name, **extra) for a in np.logspace(-4, 1, 20)]

    def dev():
        d = sglm_pp.timeshift_multiple(X0, shift_amt_list=shifts)[lo:hi]
        return sglm_cv.cv_glm_mult_params(d, y, folds, model_name, [dict(g) for g in grid], score_method="r2")
    sec, r, per = timed(dev, reps=2, warm=1)
    diag = _engine.last_poisson_batch
    return {"config": "%s: %s GLM (power %g, log link, L2) alpha sweep logspace(-4, 1, 20) x (5 folds + refit) = 120 fits, "
                      "1M timepoints x 20 predictors x 40 shifts = 800 columns, response of the family, every fit driven to "
                      "its optimum (step bound 1e-8)" % (name, model_name, power),
            "fits": 120, "seconds": sec, "fits_per_s": 120 / sec, "best_params": r["best_params"], "batch": diag,
            "rounds": diag[0]["rounds"] if diag else None,
            "refreshes": diag[0]["refreshes"] if diag else None,
            "n_iter_min_max": [int(min(np.min(x["_fit_info"]["n_iter"]) for x in r["full_cv_results"])),
                               int(max(np.max(x["_fit_info"]["n_iter"]) for x in r["full_cv_results"]))],
            "per_entry_ms": per}


def run_c4en(cpu):
    """c4 (Poisson response, design, folds) with elastic-net sets: no CPU baseline (scikit-learn has no L1 Poisson)."""
    X0_h, X0, shifts, (lo, hi), y, n = session(1_000_000, 20, -20, 19, 4, poisson=True)
    folds_h = synth_data.synth_folds(n, 5, 4)
    folds = [(torch.from_numpy(a).cuda(), torch.from_numpy(b).cuda()) for a, b in folds_h]
    grid = [dict(alpha=float(a), l1_ratio=r, model_name="Poisson") for r in (0.1, 0.5, 0.9) for a in np.logspace(-4, 1, 20)]

    def dev():
        d = sglm_pp.timeshift_multiple(X0, shift_amt_list=shifts)[lo:hi]
        return sglm_cv.cv_glm_mult_params(d, y, folds, "Poisson", [dict(g) for g in grid], score_method="r2")
    sec, r, per = timed(dev, reps=2, warm=1)
    diag = _engine.last_poisson_batch or []
    nnz = [int(np.count_nonzero(x["model"].coef_)) for x in r["full_cv_results"]]
    return {"config": "c4en: Poisson GLM (log link, elastic net) alpha sweep logspace(-4, 1, 20) x l1_ratio 0.1 / 0.5 / 0.9 x "
                      "(5 folds + refit) = 360 fits in batches of %d, 1M timepoints x 20 predictors x 40 shifts = 800 columns, "
                      "every fit driven to its optimum (step bound 1e-8)" % _engine.PB_MAX_BATCH,
            "fits": 360, "seconds": sec, "fits_per_s": 360 / sec, "best_params": r["best_params"], "batch": diag,
            "rounds": [d["rounds"] for d in diag], "refreshes": [d["refreshes"] for d in diag],
            "inner_cd_sweeps": [d.get("inner_sweeps") for d in diag],
            "refit_nonzero_min_max": [min(nnz), max(nnz)],
            "n_iter_min_max": [int(min(np.min(x["_fit_info"]["n_iter"]) for x in r["full_cv_results"])),
                               int(max(np.max(x["_fit_info"]["n_iter"]) for x in r["full_cv_results"]))],
            "per_entry_ms": per}


if __name__ == "__main__":
    which = [a for a in sys.argv[1:] if not a.startswith("--")] or ["c1", "c2", "c4"]
    cpu = "--no-cpu" not in sys.argv
    runs = {"c1": run_c1, "c2": run_c2, "c4": run_c4,
            "c4g": lambda cpu: run_c4_family("c4g", "Gamma", 2.0), "c4t": lambda cpu: run_c4_family("c4t", "Tweedie", 1.5),
            "c4en": run_c4en}
    for name in which:
        line = runs[name](cpu)
        print(json.dumps(line), flush=True)
        torch.cuda.empty_cache()
