"""torchrun --nproc-per-node N scripts/strong_glm_check.py [--reps 3] [--out profiles/NAME.jsonl] : the log-link
families on the strong-scaled multi-GPU path at the BASELINE configs[3] shape (c4: 20 alphas x (5 folds + refit) = 120
fits, 1M x 800 lag design built from 20 base signals) for Poisson, Gamma and Tweedie power 1.5, each on a response of
its family.

Per family, timed after one warm-up run, `--reps` repetitions each (min / median / max reported):
  strong  sglm_dist.cv_grid_strong on all N GPUs (rows sharded, every cross-row sum combined over the ranks)
  sharded sglm_dist.cv_glm_mult_params_sharded on the same N GPUs (parameter sets dealt to the ranks, all rows each)
  single  sglm_cv.cv_glm_mult_params on rank 0 alone
Rank 0 checks the strong grid against the one-GPU grid: best_params identical, coefficients and intercepts within
|d|_inf / |w|_inf <= 1e-7, scores within 1e-9, n_iter within +-1 — and the parameter-set route against the same bounds.  One JSON line per family (device name and power limit from a read-only nvidia-smi query, every rank's stage
timeline of the last strong run) goes to stdout and to --out."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "sabatinilab-glm_b200"), os.path.join(ROOT, "scripts")):
    sys.path.insert(0, p)
import synth_data  # noqa: E402
import sglm_cv, sglm_dist  # noqa: E402,E401
from config_bench import session  # noqa: E402

FAMILIES = [("Poisson", 1.0), ("Gamma", 2.0), ("Tweedie", 1.5)]


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True, check=False).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else "unknown"


def timed(fn, reps):
    fn()                                            # warm-up: module loads, allocator, NCCL channels
    out, secs = None, []
    for _ in range(reps):
        dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        dist.barrier()
        secs.append(time.perf_counter() - t0)
    return out, secs


def spread(secs):
    return {"min_s": min(secs), "median_s": float(np.median(secs)), "max_s": max(secs), "reps": len(secs)}


def parity(got, want):
    worst = dict(coef=0.0, icpt=0.0, score=0.0, iters=0)
    for a, b in zip(got["full_cv_results"], want["full_cv_results"]):
        for j in range(b["cv_coefs"].shape[1]):
            d = np.max(np.abs(a["cv_coefs"][:, j] - b["cv_coefs"][:, j])) / max(np.max(np.abs(b["cv_coefs"][:, j])), 1e-12)
            worst["coef"] = max(worst["coef"], float(d))
        d = np.max(np.abs(a["model"].coef_ - b["model"].coef_)) / max(np.max(np.abs(b["model"].coef_)), 1e-12)
        worst["coef"] = max(worst["coef"], float(d))
        worst["icpt"] = max(worst["icpt"], float(np.max(np.abs(a["cv_intercepts"] - b["cv_intercepts"]))),
                            abs(a["model"].intercept_ - b["model"].intercept_))
        for k in ("cv_scores_train", "cv_scores_test", "cv_mean_score", "cv_R2_score", "cv_mse_score"):
            worst["score"] = max(worst["score"], float(np.max(np.abs(np.subtract(a[k], b[k])))))
        if "_fit_info" in a and "_fit_info" in b:
            worst["iters"] = max(worst["iters"], int(np.max(np.abs(a["_fit_info"]["n_iter"].astype(np.int64) -
                                                                   b["_fit_info"]["n_iter"].astype(np.int64)))))
    ok = (got["best_params"] == want["best_params"] and worst["coef"] <= 1e-7 and worst["icpt"] <= 1e-7 and
          worst["score"] <= 1e-9 and worst["iters"] <= 1)
    return ok, worst


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    ap.add_argument("--shared-gpu", action="store_true",
                    help="every rank on GPU 0 over gloo: checks the parity of the row-sharded grid on a one-GPU box "
                         "(its times are not those of N GPUs)")
    args = ap.parse_args()
    local = 0 if args.shared_gpu else int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    if args.shared_gpu:
        dist.init_process_group("gloo")
    else:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank, world = dist.get_rank(), dist.get_world_size()
    devices = [None] * world
    dist.all_gather_object(devices, gpu_info())
    all_ok = True
    for name, power in FAMILIES:
        X0 = shifts = y = folds = d = None
        if rank == 0:
            _, X0, shifts, (lo, hi), y, n = session(1_000_000, 20, -20, 19, 4, **({"poisson": True} if power == 1 else
                                                                                  {"power": power}))
            folds = synth_data.synth_folds(n, 5, 4)
            y = y.cpu().numpy()
            import sglm_pp
            d = sglm_pp.timeshift_multiple(X0, shift_amt_list=shifts)[lo:hi]
        meta = [shifts]
        dist.broadcast_object_list(meta, src=0)
        shifts = meta[0]
        extra = {} if name in ("Poisson", "Gamma") else {"power": power}
        grid = [dict(alpha=float(a), model_name=name, **extra) for a in np.logspace(-4, 1, 20)]

        strong, t_strong = timed(lambda: sglm_dist.cv_grid_strong(X0, shifts, y, folds, name, [dict(g) for g in grid],
                                                                  score_method="r2"), args.reps)
        timelines = [None] * world
        dist.all_gather_object(timelines, sglm_dist.last_timeline)
        # the parameter-set route: every rank holds the whole design
        Xt, yt, idx = sglm_dist.broadcast_inputs(d, y, folds, src=0, device="cuda")
        sharded, t_sharded = timed(lambda: sglm_dist.cv_glm_mult_params_sharded(Xt, yt, idx, name, [dict(g) for g in grid],
                                                                                score_method="r2"), args.reps)
        del Xt, yt, idx
        line = {"family": name, "power": power, "ranks": world, "shared_gpu": args.shared_gpu, "devices": devices,
                "shape": "1M x 800 (20 base signals x 40 shifts), 20 alphas x (5 folds + refit) = 120 fits",
                "strong": spread(t_strong), "sharded": spread(t_sharded), "strong_timeline_ms": timelines}
        if rank == 0:
            t_single = []
            single = sglm_cv.cv_glm_mult_params(d, y, folds, name, [dict(g) for g in grid], score_method="r2")
            for _ in range(args.reps):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                single = sglm_cv.cv_glm_mult_params(d, y, folds, name, [dict(g) for g in grid], score_method="r2")
                torch.cuda.synchronize()
                t_single.append(time.perf_counter() - t0)
            ok, worst = parity(strong, single)
            ok_sh, worst_sh = parity(sharded, single)
            line.update(single=spread(t_single), parity_strong_vs_single=worst, parity_ok=bool(ok),
                        sharded_vs_single=worst_sh, best_params=strong["best_params"])
            all_ok = all_ok and ok and ok_sh
            print(json.dumps(line), flush=True)
            if args.out:
                with open(args.out, "a") as f:
                    f.write(json.dumps(line) + "\n")
        dist.barrier()
        del d, X0
    flag = torch.tensor([int(all_ok)], device="cuda")
    dist.broadcast(flag, src=0)
    if rank == 0:
        print("STRONG GLM CHECK " + ("OK" if int(flag.item()) else "FAILED"), flush=True)
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if int(flag.item()) else 1)


if __name__ == "__main__":
    main()
