"""
bench.py — CV model fits/sec of the sGLM hot path on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W          (N>1: launched by torch.distributed.run)
    python bench.py --impl reference ...                   (CPU arm: the reference's own path)
    python bench.py ... --dump-outputs DIR                 (also write the last timed step's results as DIR/*.npy)

One "step" = one pass of the hot path over one synthetic session:
    lag/shift gather  (T x P base signals  ->  T x C design, NaN edge rows dropped)
 -> CV grid of penalised Gaussian GLM fits: n_sets x (n_folds + 1) fits, the count the
    reference performs in cv_glm_mult_params (backend/sglm_cv.py:210-428).
Workload (default) = BASELINE.json configs[2], the configuration the north-star target is
quoted on and the largest that fits one GPU: ElasticNet grid 5 folds x 50 alphas x 5
l1_ratios on a 2M-timepoint x 2000-column lagged design (P=40 base signals x 50 shifts).

`value`  : device-resident throughput (base signals, response, fold indices already in HBM).
`e2e`    : the same step through the reference-facing API with HOST buffers — numpy base signals,
           numpy response, numpy fold index lists in; result dicts of numpy arrays out
           (sglm_pp.timeshift_multiple(..., device=True).dropna() -> sglm_cv.cv_glm_mult_params).

Multi-GPU (--mode):
    grid     (default)  ONE grid strong-scaled over the N GPUs: base signals broadcast, every rank gathers its
                        row slice locally and multiplies its rows of the Gram (exact int64 all-reduce), the
                        models are dealt to the ranks by cost, results come back in one packed all_gather.
    sessions            one independent session per rank (BASELINE configs[4]), weak scaling, no collective.
Timing = CUDA events, barrier + synchronize on both sides, max over ranks.
"""
import os
import sys

if "--impl" in sys.argv and "reference" in sys.argv:
    # the CPU arm uses every host core whatever the launcher exported (torchrun sets OMP_NUM_THREADS=1)
    _n = str(len(os.sched_getaffinity(0)))
    for _k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[_k] = _n

import argparse
import json
import subprocess
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "sabatinilab-glm_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

import synth_data  # noqa: E402

METRIC = "cv_model_fits_per_sec"
UNIT = "fits/s"
FALLBACK_PEAKS = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3, help="timed steps of every timed leg (device-resident, end to end, "
                                                         "--impl reference); the cpu_baseline leg times one sample step")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--mode", default="grid", choices=["grid", "sessions"])
    ap.add_argument("--sessions-per-gpu", type=int, default=1,
                    help="sessions mode: independent sessions batched into one launch plan per GPU (BASELINE configs[4]: "
                         "64 sessions on 8 GPUs = 8 per GPU at --T 250000)")
    ap.add_argument("--T", type=int, default=2_000_000)
    ap.add_argument("--P", type=int, default=40)
    ap.add_argument("--shift-lo", type=int, default=-20)
    ap.add_argument("--shift-hi", type=int, default=29)
    ap.add_argument("--folds", type=int, default=5)
    ap.add_argument("--alphas", type=int, default=50)
    ap.add_argument("--l1s", type=int, default=5)
    ap.add_argument("--max-iter", type=int, default=1000)
    ap.add_argument("--tol", type=float, default=1e-4)
    ap.add_argument("--warm-path", action="store_true",
                    help="opt-in non-reference mode: warm-started alpha paths (NOT the parity configuration)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-probes", action="store_true")
    ap.add_argument("--cpu-sample-T", type=int, default=0, help="rows of the CPU sample (0: 40000 for --impl reference, "
                                                               "16000 for the cpu_baseline leg)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last device-resident step returned (per parameter set: "
                         "fold and refit coefficients, intercepts, scores; the selection) as DIR/<name>.npy in float64, "
                         "at most 64 MB (a seeded sample of the parameter sets beyond that)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def workload(args):
    shifts = [0] + [s for s in range(args.shift_lo, args.shift_hi + 1) if s != 0]
    alphas = np.logspace(-4, 0, args.alphas)
    l1s = np.linspace(0.1, 0.9, args.l1s) if args.l1s > 1 else np.array([0.5])
    grid = [dict(alpha=float(a), l1_ratio=float(round(l, 6)), max_iter=args.max_iter, fit_intercept=True,
                 tol=args.tol) for l in l1s for a in alphas]
    return shifts, grid


def make_session(args, seed, T):
    """Host-side synthetic session: base signals, kernels, noise, folds (design built later)."""
    shifts, _ = workload(args)
    X0 = synth_data.synth_base(T, args.P, seed)
    beta = synth_data.synth_kernels(args.P, shifts, seed)
    h_lo, h_hi = max(0, max(shifts)), max(0, -min(shifts))     # NaN rows at the top / bottom
    n_valid = T - h_lo - h_hi
    folds = synth_data.synth_folds(n_valid, args.folds, seed, group=1000)
    return X0, beta, (h_lo, h_hi), folds


def config_dict(args, n_gpus, mode):
    shifts, grid = workload(args)
    C = args.P * len(shifts)
    spg = getattr(args, "sessions_per_gpu", 1)
    layout = ("ONE grid strong-scaled over the GPUs (row-sharded Gram + models dealt by cost)" if mode == "grid"
              else f"{spg} independent session(s) per GPU, batched into one launch plan per GPU (BASELINE.json configs[4])")
    return {"workload": f"ElasticNet CV grid {args.folds} folds x {args.alphas} alphas x {args.l1s} l1_ratios "
                        f"(+1 full-data refit per set = {len(grid) * (args.folds + 1)} fits/step) on "
                        f"{args.T} timepoints x {C} lagged columns (P={args.P} base signals x {len(shifts)} shifts), "
                        f"fp64, tol={args.tol}, max_iter={args.max_iter}, "
                        f"{'WARM-STARTED alpha paths (non-reference mode)' if args.warm_path else 'cold start'}, cyclic CD "
                        f"(BASELINE.json configs[2]); {layout}",
            "T": args.T, "C": C, "folds": args.folds, "alphas": args.alphas, "l1_ratios": args.l1s,
            "fits_per_step": len(grid) * (args.folds + 1), "mode": mode,
            "sessions": n_gpus * spg if mode == "sessions" else 1,
            "l2_policy": ("inputs and working set larger than L2: base signals %.2f GB in, int8 digit planes of the %.0f GB design "
                          "(~%.1f GB) written and re-read by the Gram GEMM, 6 x %.0f MB centred statistics streamed by coordinate "
                          "descent (126 MB L2); the fp64 design itself is never built on the statistics path"
                          % (args.T * args.P * 8 / 1e9, args.T * C * 8 / 1e9, args.T * C * 2.4 / 1e9, C * C * 8 / 1e6)),
            "host": "Python cyclic GC frozen after the warm-up steps (gc.freeze): a generation-2 pass over the interpreter's "
                    "module objects is ~50 ms of host time"}


# --------------------------------------------------------------------------- #
# clocks sampling during the timed region
# --------------------------------------------------------------------------- #
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", os.environ.get("BENCH_SAMPLER_MS", "200")],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        self.thread.join(timeout=2)
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(len(r) >= 6 and r[2 + k] == "Active" for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# --------------------------------------------------------------------------- #
# CPU arm: the reference's path on host cores (oracle port, scikit-learn numerics)
# --------------------------------------------------------------------------- #
def cpu_reference_run(args, Ts, strata, n_folds, steps, warmup):
    """Times the reference's CPU path — oracle restatement of backend/sglm_pp.py + backend/sglm_cv.py +
    backend/sglm.py handing each fit to the installed scikit-learn (exactly what the reference executes), fold
    fits on up to 4 threads as in backend/sglm_cv.py:162-170, BLAS/OpenMP on all host cores — on a BOUNDED,
    STRATIFIED sample of the workload and extrapolates to the full workload:

      sample  : the parameter sets at `strata` alpha positions (the smallest alpha — the slowest fits — always
                included) x the middle l1_ratio, each with (n_folds folds + refit) on Ts of the T timepoints,
                timed per set, plus the host lag gather + dropna once per step;
      full    : seconds(full grid, T rows) = (T / Ts) * rounds_full / rounds_sample * n_l1 *
                sum over all alphas of t(alpha), t() interpolated linearly in the alpha index between the
                strata; rounds = ceil(folds / 4) + 1 fit-times per set with the reference's 4 fold threads.
                Per-fit cost of coordinate descent is linear in the rows (two passes over X per sweep, the
                number of sweeps does not depend on n), and at full size X (32 GB) no longer fits any cache,
                so the extrapolation favours the CPU.
    Returns (full-size fits/s, sample fits/s, seconds per step, description)."""
    from oracle import sglm_oracle as orc
    import warnings
    warnings.filterwarnings("ignore")
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=len(os.sched_getaffinity(0)))
    except Exception:
        pass
    shifts, grid = workload(args)
    A, R = args.alphas, args.l1s
    Ts = min(Ts, args.T)
    X0 = synth_data.synth_base(Ts, args.P, 1234)
    beta = synth_data.synth_kernels(args.P, shifts, 1234)
    pos = sorted({int(round(f * (A - 1))) for f in strata})
    l1_mid = R // 2
    step_secs, per_set = [], None
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        Xd = orc.timeshift_multiple(X0, shift_amt_list=shifts)
        Xd = Xd[~np.isnan(Xd).any(axis=1)]
        t_gather = time.perf_counter() - t0
        if it == 0:
            y = synth_data.synth_response(Xd, beta, 1234)
            folds = synth_data.synth_folds(Xd.shape[0], n_folds, 1234, group=1000)
        secs = []
        for a_i in pos:
            t1 = time.perf_counter()
            orc.cv_glm_mult_params(Xd, y, folds, "Gaussian", [dict(grid[l1_mid * A + a_i])], score_method="r2",
                                   engine="sklearn", n_threads=4)
            secs.append(time.perf_counter() - t1)
        if it >= warmup:
            step_secs.append(time.perf_counter() - t0)
            per_set = np.array(secs) if per_set is None else per_set + np.array(secs)
    per_set = per_set / max(1, steps)
    sec = float(np.mean(step_secs))
    fits_sample = len(pos) * (n_folds + 1)
    rounds_sample = -(-n_folds // 4) + 1
    rounds_full = -(-args.folds // 4) + 1
    t_all = np.interp(np.arange(A), pos, per_set)
    full_seconds = (args.T / Ts) * (rounds_full / rounds_sample) * R * float(t_all.sum()) + t_gather * (args.T / Ts)
    full_value = len(grid) * (args.folds + 1) / full_seconds
    C = args.P * len(shifts)
    sample = (f"stratified sample: alpha positions {pos} of {A} x l1_ratio {grid[l1_mid * A]['l1_ratio']} "
              f"x ({n_folds} folds + refit) = {fits_sample} sklearn ElasticNet fits on {Ts} of {args.T} timepoints x {C} "
              f"columns, {sec:.1f} s per step (per set: {[round(float(s), 2) for s in per_set]} s), incl. the host lag "
              f"gather; `value` = extrapolation to the full grid at full T (x{args.T / Ts:.0f} rows, alpha positions "
              f"interpolated, {rounds_full}/{rounds_sample} fit rounds per set) = {full_seconds:.0f} s per grid; "
              f"scikit-learn {__import__('sklearn').__version__}, 4 fold threads")
    return full_value, fits_sample / sec, sec, sample, dict(sample_T=Ts, alpha_positions=pos, n_folds=n_folds,
                                                              sample_fits=fits_sample, seconds_per_set=per_set.tolist(),
                                                              full_grid_seconds_extrapolated=full_seconds)


# --------------------------------------------------------------------------- #
def measure_probes(nat, torch):
    """Measured denominators of this run: L2 -> SM read bandwidth (32 MB buffer, the size of one Gram matrix),
    HBM read bandwidth (4 GB buffer), tcgen05 kind::i8 issue rate."""
    out = {}
    sink = torch.zeros(1, dtype=torch.float64, device="cuda")
    st = nat.stream_ptr()

    def timed(fn, reps=3):
        best = None
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            best = ms if best is None else min(best, ms)
        return best
    small = torch.ones(4 * 1024 * 1024, dtype=torch.float64, device="cuda")          # 32 MB
    nat.lib().sglm_probe_read_f64(nat.ptr(small), small.numel(), 20, 8, nat.ptr(sink), st)
    ms = timed(lambda: nat.lib().sglm_probe_read_f64(nat.ptr(small), small.numel(), 400, 8, nat.ptr(sink), st))
    out["l2_read_gbs"] = small.numel() * 8 * 400 / ms / 1e6
    big = torch.ones(512 * 1024 * 1024, dtype=torch.float64, device="cuda")          # 4 GB
    ms = timed(lambda: nat.lib().sglm_probe_read_f64(nat.ptr(big), big.numel(), 2, 8, nat.ptr(sink), st))
    out["hbm_read_gbs"] = big.numel() * 8 * 2 / ms / 1e6
    del big, small
    import ctypes
    n_ctas = ctypes.c_int64(0)
    nat.lib().sglm_probe_mma_i8(2000, ctypes.byref(n_ctas), st)
    iters = 40000
    ms = timed(lambda: nat.lib().sglm_probe_mma_i8(iters, ctypes.byref(n_ctas), st))
    out["mma_i8_tops"] = 2.0 * n_ctas.value * iters * 8 * 128 * 256 * 32 / ms / 1e9
    out["how"] = ("sglm_probe_read_f64 (16-byte loads, 8 in flight per thread, 8 CTAs/SM) on a 32 MB / 4 GB buffer; "
                  "sglm_probe_mma_i8: tcgen05.mma kind::i8 M128 N256 K32 issued back to back from shared memory, "
                  "one CTA per SM; best of 3, CUDA events")
    return out


DUMP_LIMIT_BYTES = 64 * 2**20
DUMP_FIELDS = ("cv_coefs", "cv_intercepts", "cv_scores_train", "cv_scores_test", "cv_mean_score_train", "cv_mean_score",
               "cv_std_score", "cv_R2_score", "cv_mse_score")


def dump_outputs(res, out_dir):
    """Writes the result dict of one CV grid step as float64 DIR/<name>.npy, row i = parameter set set_index[i] of the
    grid: the DUMP_FIELDS of every set (cv_coefs stacked to sets x C x folds), the refit's coef / intercept, and the
    selection (best_set, best_score, best_score_std).  Two builds run with the same arguments get the same inputs, so
    their dumps compare output for output.  Past DUMP_LIMIT_BYTES a fixed, seeded sample of the sets is written."""
    full = res["full_cv_results"]

    def row(r):
        return [r[k] for k in DUMP_FIELDS] + [r["model"].coef_, r["model"].intercept_]
    names = list(DUMP_FIELDS) + ["coef", "intercept"]
    n = len(full)
    row_bytes = 8 * (1 + sum(np.size(v) for v in row(full[0])))       # + its set_index entry
    k = min(n, (DUMP_LIMIT_BYTES - 4096) // row_bytes)
    idx = np.arange(n) if k == n else np.sort(np.random.default_rng(0).choice(n, k, replace=False))
    rows = [row(full[i]) for i in idx]
    out = {name: np.stack([np.asarray(r[j], dtype=np.float64) for r in rows]) for j, name in enumerate(names)}
    out["set_index"] = idx.astype(np.float64)
    out["best_set"] = np.float64([r["glm_kwargs"] for r in full].index(res["best_params"]))
    out["best_score"] = np.float64(res["best_score"])
    out["best_score_std"] = np.float64(res["best_score_std"])
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    mb = sum(a.nbytes for a in out.values()) / 2**20
    sys.stderr.write(f"[dump] {len(out)} arrays, {mb:.1f} MB, {k} of {n} parameter sets -> {out_dir}\n")


def main():
    args = parse_args()
    # stdout carries exactly ONE JSON line: everything else written to file descriptor 1 by libraries (NCCL prints its
    # version banner there) goes to stderr
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(line):
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    n_gpus = max(args.gpus, world)
    cores = len(os.sched_getaffinity(0))
    mode = args.mode

    if args.impl == "reference":
        if rank != 0:
            return
        steps, warmup = args.steps, min(args.warmup, 1)
        Ts = args.cpu_sample_T or 40_000
        v, v_sample, sec, sample, detail = cpu_reference_run(args, Ts, (0.0, 0.25, 0.5, 1.0), 3, steps, warmup)
        cfg = config_dict(args, n_gpus, mode)
        cfg["reference_sample"] = detail
        line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": n_gpus, "steps": steps,
                "warmup": warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
                "scaling": "strong" if mode == "grid" else "weak",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": cfg,
                "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                                 "sample_value": v_sample},
                "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        emit(line)
        return

    import torch
    import torch.distributed as dist
    import _sglm_native as nat
    import sglm_cv
    import sglm_pp
    import _engine
    _engine.WARM_START_PATHS = bool(args.warm_path)

    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    shifts, grid = workload(args)
    C = args.P * len(shifts)
    fits_per_step = len(grid) * (args.folds + 1)
    strong = mode == "grid" and world > 1

    # ---- synthetic session (host): one per rank in `sessions` mode, ONE (rank 0's) in `grid` mode
    seed = 1234 + (rank if mode == "sessions" else 0)
    X0_h, beta, (h_lo, h_hi), folds_h = make_session(args, seed, args.T)
    X0_pin = torch.from_numpy(X0_h).pin_memory()
    X0_d = X0_pin.to("cuda")
    design = sglm_pp.timeshift_multiple(X0_d, shift_amt_list=shifts)
    Xv = design[h_lo: args.T - h_hi]
    noise_seed = 99 + (rank if mode == "sessions" else 0)
    s = Xv @ torch.from_numpy(beta).cuda()                      # data generation only (not timed)
    from scipy.signal import lfilter
    e = lfilter([1.0], [1.0, -0.95], np.random.default_rng(noise_seed).standard_normal(Xv.shape[0]))
    e = torch.from_numpy(e / e.std()).cuda() * s.std() * float(np.sqrt(0.7 / 0.3))
    y_d = s + e
    y_d = ((y_d - y_d.mean()) / y_d.std()).contiguous()
    y_pin = y_d.cpu().pin_memory()
    del s, e, design, Xv
    folds_pin = [(torch.from_numpy(a).pin_memory(), torch.from_numpy(b).pin_memory()) for a, b in folds_h]
    folds_d = [(a.to("cuda"), b.to("cuda")) for a, b in folds_pin]
    # host views for the end-to-end leg: plain numpy arrays (what a reference user holds), backed by pinned memory
    X0_np, y_np = X0_pin.numpy(), y_pin.numpy()
    folds_np = [(a.numpy(), b.numpy()) for a, b in folds_pin]
    torch.cuda.synchronize()

    extra_sessions = []
    if mode == "sessions" and args.sessions_per_gpu > 1:
        # BASELINE configs[4]: several independent sessions per GPU, all their models in one launch plan
        def one_session(seed_i):
            X0_i, beta_i, _, folds_i = make_session(args, seed_i, args.T)
            X0_di = torch.from_numpy(X0_i).cuda()
            Xi = sglm_pp.timeshift_multiple(X0_di, shift_amt_list=shifts)[h_lo: args.T - h_hi]
            si = Xi @ torch.from_numpy(beta_i).cuda()
            gi = torch.Generator(device="cuda").manual_seed(seed_i)
            yi = si + float(si.std()) * float(np.sqrt(0.7 / 0.3)) * torch.randn(si.shape, dtype=torch.float64, device="cuda", generator=gi)
            yi = ((yi - yi.mean()) / yi.std()).contiguous()
            return X0_di, yi, [(torch.from_numpy(a).cuda(), torch.from_numpy(b).cuda()) for a, b in folds_i]
        extra_sessions = [one_session(5000 + rank * args.sessions_per_gpu + i) for i in range(1, args.sessions_per_gpu)]

    if strong:
        import sglm_dist

        def step_device():
            return sglm_dist.cv_grid_strong(X0_d if rank == 0 else None, shifts, y_d if rank == 0 else None,
                                            folds_d if rank == 0 else None, "Gaussian", [dict(g) for g in grid],
                                            score_method="r2", rows=(h_lo, args.T - h_hi))

        def step_e2e():
            return sglm_dist.cv_grid_strong(X0_np if rank == 0 else None, shifts, y_np if rank == 0 else None,
                                            folds_np if rank == 0 else None, "Gaussian", [dict(g) for g in grid],
                                            score_method="r2", rows=(h_lo, args.T - h_hi))
    elif extra_sessions:
        def step_device():
            ses = [(sglm_pp.timeshift_multiple(x0, shift_amt_list=shifts, device=True).dropna(), yy, ff)
                   for x0, yy, ff in [(X0_d, y_d, folds_d)] + extra_sessions]
            return sglm_cv.cv_glm_mult_params_sessions(ses, "Gaussian", [dict(g) for g in grid], score_method="r2")[0]
        step_e2e = None
    else:
        def step_device():
            # inputs resident in HBM; the design stays a recipe (base signals + column map + valid rows): the grid's
            # statistics are computed from the base signals, the 32 GB design is never built (DESIGN.md section 4)
            d = sglm_pp.timeshift_multiple(X0_d, shift_amt_list=shifts, device=True).dropna()
            return sglm_cv.cv_glm_mult_params(d, y_d, folds_d, "Gaussian", [dict(g) for g in grid], score_method="r2")

        def step_e2e():
            # the reference-facing call sequence with HOST buffers (numpy in, numpy result dicts out)
            d = sglm_pp.timeshift_multiple(X0_np, shift_amt_list=shifts, device=True).dropna()
            return sglm_cv.cv_glm_mult_params(d, y_np, folds_np, "Gaussian", [dict(g) for g in grid], score_method="r2")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        res = None
        for _ in range(steps):
            res = fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), res

    probes = None
    if rank == 0 and not args.no_probes:
        probes = measure_probes(nat, torch)
    for _ in range(args.warmup):
        res = step_device()
    # Python's cyclic collector: a generation-2 pass walks every live object of the interpreter (torch, pandas, scipy
    # modules: ~50 ms, measured with gc.callbacks) and lands in a timed step now and then.  Objects alive after the
    # warm-up are moved to the permanent generation, so later passes only walk what the steps themselves allocate.
    import gc
    gc.collect()
    gc.freeze()
    gc_log = []
    if os.environ.get("BENCH_GAPS"):
        t_gc = [0.0]

        def _gc_cb(phase, info):
            if phase == "start":
                t_gc[0] = time.perf_counter()
            else:
                gc_log.append((info.get("generation"), round((time.perf_counter() - t_gc[0]) * 1e3, 2)))
        gc.callbacks.append(_gc_cb)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = nat.launches()
    nat.enable_timing(True)
    nat.collect_timing()
    _engine.CD_COLLECT_STATS = True
    _engine.cd_parts_log.clear()
    total_ms, res = timed(step_device, args.steps)
    device_timeline = dict(getattr(sglm_dist, "last_timeline", None) or {}) if strong else None
    per_entry = nat.collect_timing()
    if rank == 0 and os.environ.get("BENCH_GAPS"):
        # diagnostics: where the stream idles between ABI calls (host work, read-backs, torch glue)
        iv = sorted(nat.last_intervals, key=lambda t: t[1])
        gaps, prev_end, prev_name = [], 0.0, "start"
        for name, a, b in iv:
            if a - prev_end > 0.5:
                gaps.append((round(a - prev_end, 2), prev_name, name, round(a, 1)))
            if b > prev_end:
                prev_end, prev_name = b, name
        sys.stderr.write(f"[gc] collections during the timed steps (generation, ms): {[g for g in gc_log if g[1] > 0.5]}\n")
        sys.stderr.write(f"[gaps] total {total_ms:.1f} ms, last call ends {prev_end:.1f} ms after the first; gaps > 0.5 ms: "
                         f"{sorted(gaps, reverse=True)[:12]}\n")
    cd_parts_stats = _engine.cd_stats()
    _engine.CD_COLLECT_STATS = False
    nat.enable_timing(False)
    launches = nat.launches() - launches0
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0 and args.dump_outputs:
        dump_outputs(res, args.dump_outputs)
    n_sessions = world * args.sessions_per_gpu if mode == "sessions" else 1
    value = fits_per_step * args.steps * n_sessions / (total_ms / 1e3)

    # ---- per-kernel accounting for the roofline of the dominant kernel (rank 0's launches)
    peaks = dict(FALLBACK_PEAKS)
    peaks_src = "fallback (B200_PROFILING.md)"
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks.update(json.load(f))
            peaks_src = "MEASURED_PEAKS.json"
    except Exception:
        pass
    tc_plan = nat.last_tc_plan
    n_rows = args.T - h_lo - h_hi
    n_test = sum(len(b) for _, b in folds_h)
    n_aug = C + 2
    k_ms = {name: ms / args.steps for name, (calls, ms) in per_entry.items()}
    # the coordinate-descent grid is one logical kernel: its parts (clusters of heavy models, one CTA per
    # light model) are launched on two streams and overlap, so the time they cover together is what counts
    cd_names = ("sglm_enet_cd_cluster_f64", "sglm_enet_cd_gram_f64")
    cd_part_ms = {n: k_ms.pop(n) for n in cd_names if n in k_ms}
    # per LAUNCH of a step (a plan may hold several cluster launches): launch order inside a step = plan order
    cd_launch_ms = []
    for n in cd_names:
        iv = sorted((a, b) for nm, a, b in nat.last_intervals if nm == n)
        per_step = len(iv) // max(1, args.steps)
        for j in range(per_step):
            sel = iv[j::per_step] if per_step else []
            cd_launch_ms.append((n, j, sum(b - a for a, b in sel) / max(1, len(sel))))
    CD = "sglm_enet_cd (cluster + per-model parts, concurrent)" if len(cd_part_ms) > 1 else next(iter(cd_part_ms), cd_names[0])
    if cd_part_ms:
        k_ms[CD] = nat.union_ms(cd_names) / args.steps
    for a, b in (("sglm_gram_tc_cells_f64", "sglm_gram_tc_f64"), ("sglm_gram_tc_cells_partial_f64", "sglm_gram_tc_f64"),
                 ("sglm_gram_tc_lag_cells_f64", "sglm_gram_tc_f64"), ("sglm_gram_tc_cells_combine_f64", "sglm_gram_tc_f64")):
        if a in k_ms:
            k_ms[b] = k_ms.get(b, 0.0) + k_ms.pop(a)
    dominant = max(k_ms, key=k_ms.get)
    step_ms = total_ms / args.steps
    hbm_peak = peaks["hbm_gbs"]
    # coordinate descent: what the SMs pulled through L2 (rows of Q: 8*C bytes each, a moved row once per cluster
    # group — counted by the kernels — plus q, diag, w per sweep), the coordinate updates it stands for
    # (8*C "algorithmic" bytes each: what a one-model-at-a-time solver would stream), and the serial chain
    n_steps_logged = max(1, args.steps)
    rows_loaded = sum(p["rows_loaded"] for p in cd_parts_stats) / n_steps_logged
    n_upd = sum(p["row_updates"] for p in cd_parts_stats) / n_steps_logged
    full = res["full_cv_results"] if res is not None else []
    n_sweeps = float(sum(np.sum(r["_fit_info"]["cd_info"][:, 2]) for r in full if "_fit_info" in r))
    n_unconv = int(sum(np.sum(r["_fit_info"]["status"] != 0) for r in full if "_fit_info" in r))
    cd_sec = k_ms.get(CD, float("nan")) / 1e3
    l2_bytes = rows_loaded * 8.0 * C + n_sweeps * 8.0 * 3 * C
    traffic_tbl = {}
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            traffic_tbl = json.load(f)
    except Exception:
        pass

    def dram_traffic(key, scale_by=None):
        tr = traffic_tbl.get(key, {})
        if scale_by is not None and tr.get("dram_bytes_per_row_update"):
            return tr["dram_bytes_per_row_update"] * scale_by
        return tr.get("dram_bytes_per_launch")

    heaviest = max((p for p in cd_parts_stats), key=lambda p: p["max_blocks_one_model"], default=None)
    chain = None
    if heaviest:
        # the launch that holds the heaviest model: cluster launches are logged in plan order, the per-model launch last
        cl = [p for p in cd_parts_stats[:max(1, len(cd_parts_stats) // max(1, args.steps))] if p["shape"] != "0x0"]
        if heaviest["shape"] != "0x0":
            j = next((k for k, p in enumerate(cl) if p["shape"] == heaviest["shape"]), 0)
            part_ms = next((ms for n, jj, ms in cd_launch_ms if n == "sglm_enet_cd_cluster_f64" and jj == j), float("nan"))
        else:
            part_ms = next((ms for n, jj, ms in cd_launch_ms if n == "sglm_enet_cd_gram_f64"), float("nan"))
        chain = {"heaviest_model_blocks": heaviest["max_blocks_one_model"], "heaviest_model_sweeps": heaviest["max_sweeps"],
                 "its_part": heaviest["shape"], "its_part_ms": part_ms,
                 "us_per_block_if_chain_bound": part_ms * 1e3 / max(1.0, heaviest["max_blocks_one_model"]),
                 "register_phase_share_of_that_model": heaviest["register_phase_share_heaviest"],
                 "note": "a model is a serial chain of 32-coordinate blocks (register phase -> record -> panel); the "
                         "part's time / the longest chain = us per block the heaviest model would need if it alone "
                         "bounded the part (measured under load: 4.0 us on (4,4), 6.1 us on (4,2), profiles/r2_cd_experiments.txt); "
                         "its_part_ms = duration of the launch that holds it (launches of a plan overlap)"}
    rooflines = {}
    l2_peak = probes["l2_read_gbs"] if probes else None
    cd_traffic = dram_traffic("sglm_enet_cd", n_upd)
    rooflines[CD] = {"kernel": CD, "bound": "latency/L2", "achieved": l2_bytes / cd_sec / 1e9, "peak": l2_peak,
                     "unit": "GB/s", "frac": (l2_bytes / cd_sec / 1e9 / l2_peak) if l2_peak else None,
                     "traffic": cd_traffic,
                     "dram_frac": (cd_traffic / cd_sec / 1e9 / hbm_peak) if cd_traffic else None,
                     "peak_source": "measured in this run: sglm_probe_read_f64 on a 32 MB (L2-resident) buffer",
                     "l2_bytes_per_step": l2_bytes, "rows_loaded_per_step": rows_loaded,
                     "coordinate_updates_per_step": n_upd, "sweeps_total": n_sweeps, "models_not_converged": n_unconv,
                     "algorithmic_GBps_one_model_at_a_time": (n_upd * 8.0 * C + n_sweeps * 8.0 * 5 * C) / cd_sec / 1e9,
                     "chain": chain, "parts": cd_parts_stats, "parts_ms_per_step": cd_part_ms,
                     "launch_ms": [{"entry": n, "launch_in_step": j, "ms": ms} for n, j, ms in cd_launch_ms],
                     "plan": _engine._cd_plan(C, fits_per_step if not strong else -(-fits_per_step // world), args.folds + 1),
                     "note": "not an HBM-bound kernel: the 6 centred Gram matrices (32 MB each) are streamed from L2 "
                             "(hit rate ~70 %), no unit is saturated (ncu: lts 20 %, fp64 17 %, DRAM 14 %); the bound is "
                             "the serial register-phase chain of the heaviest models next to the SM time of the light "
                             "ones.  achieved = bytes the SMs pulled through L2 (counted by the kernels) / time covered "
                             "by the two concurrent launches; peak = measured L2 read bandwidth"}
    gather_bytes = 8.0 * args.T * args.P + 8.0 * args.T * C
    gather_note = None
    if "sglm_timeshift_f64_ranged" not in k_ms and rank == 0:
        # the CV grid computes its statistics from the base signals (lag recipe): the design is not built inside the
        # step any more.  The gather (north_star piece 1) is measured on its own: the call a user makes to GET the design
        torch.cuda.synchronize()
        best = None
        for _ in range(3):
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            g0.record()
            dm = sglm_pp.timeshift_multiple(X0_d, shift_amt_list=shifts)
            g1.record()
            torch.cuda.synchronize()
            del dm
            best = g0.elapsed_time(g1) if best is None else min(best, g0.elapsed_time(g1))
        k_gather_ms = best
        gather_note = ("measured standalone (best of 3 calls of sglm_pp.timeshift_multiple on the resident base signals, "
                       "CUDA events): the CV step no longer builds the design")
    else:
        k_gather_ms = k_ms.get("sglm_timeshift_f64_ranged")
    if k_gather_ms:
        g_sec = k_gather_ms / 1e3
        rooflines["sglm_timeshift_f64_ranged"] = {
            "kernel": "timeshift_staged_kernel", "bound": "hbm", "achieved": gather_bytes / g_sec / 1e9, "peak": hbm_peak,
            "unit": "GB/s", "frac": gather_bytes / g_sec / 1e9 / hbm_peak, "traffic": dram_traffic("sglm_timeshift_f64_ranged"),
            "peak_source": peaks_src, "ms": k_gather_ms}
        if gather_note:
            rooflines["sglm_timeshift_f64_ranged"]["note"] = gather_note
    if "sglm_gram_tc_f64" in k_ms and tc_plan:
        t_sec = k_ms["sglm_gram_tc_f64"] / 1e3
        useful = float(n_rows + n_test) * (n_aug * (n_aug + 1.0))
        issued = 2.0 * tc_plan["tiles"] * 256 * 256 * tc_plan["n_pos"]
        gemm_ms = traffic_tbl.get("tc_gram_i8_kernel", {}).get("duration_ms")
        rooflines["sglm_gram_tc_f64"] = {
            "kernel": ("tc_slice(base signals) + tc_expand + tc_gram_i8 + tc_cell_sum + tc_combine (one entry point; lag design: "
                       "digit planes from the base signals, the fp64 design is never built)" if tc_plan.get("lag") else
                       "tc_slice + tc_gram_i8 + tc_cell_sum + tc_combine (one entry point)"), "bound": "tensor",
            "achieved": issued / t_sec / 1e12, "peak": (probes or {}).get("mma_i8_tops"), "unit": "int8 TOP/s issued",
            "frac": (issued / t_sec / 1e12 / probes["mma_i8_tops"]) if probes else None,
            "useful_fp64_equivalent_TFLOPs_syrk_honest": useful / t_sec / 1e12,
            "useful_vs_bf16_sustained_peak": useful / t_sec / 1e12 / peaks["bf16_tflops_sustained"],
            "gemm_kernel_alone": ({"ms": gemm_ms, "issued_TOPs": issued / (gemm_ms / 1e3) / 1e12,
                                   "frac_of_measured_i8_issue_rate": issued / (gemm_ms / 1e3) / 1e12 / probes["mma_i8_tops"]}
                                  if gemm_ms and probes else None),
            "traffic": dram_traffic("tc_gram_i8_kernel"), "plan": tc_plan,
            "peak_source": "measured in this run: sglm_probe_mma_i8 (tcgen05.mma kind::i8 issue rate)"}
    roofline = dict(rooflines.get(dominant, {"kernel": dominant, "bound": "hbm", "achieved": None, "peak": hbm_peak,
                                             "unit": "GB/s", "frac": None, "traffic": None}))
    roofline["share_of_step"] = k_ms[dominant] / step_ms
    roofline["per_entry_ms_per_step"] = k_ms
    roofline["other_kernels"] = {k: v for k, v in rooflines.items() if k != dominant}
    roofline["measured_peaks_this_run"] = probes
    roofline["hbm_peak_source"] = peaks_src

    # ---- end to end through the reference-facing API from host (numpy) buffers
    e2e = None
    if not args.no_e2e and step_e2e is not None:
        step_e2e()
        e2e_steps = args.steps
        e2e_ms, res_e = timed(step_e2e, e2e_steps)
        h2d = X0_pin.numel() * 8 + y_pin.numel() * 8 + sum((a.numel() + b.numel()) * 8 for a, b in folds_pin)
        d2h = 0
        if res_e is not None:
            d2h = sum(r["cv_coefs"].nbytes + r["cv_intercepts"].nbytes + r["cv_scores_train"].nbytes
                      + r["cv_scores_test"].nbytes + r["model"].coef_.nbytes + 8 * 6 for r in res_e["full_cv_results"])
        e2e = {"value": fits_per_step * e2e_steps * n_sessions / (e2e_ms / 1e3), "unit": UNIT,
               "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "steps": e2e_steps,
               "inputs": "numpy float64 base signals + response + int64 fold index lists (pinned host memory)",
               "outputs": "reference result dicts (numpy arrays)",
               "api": ("sglm_dist.cv_grid_strong(X0, shifts, y, cv_idx, ...) on rank 0's host arrays" if strong else
                       "sglm_pp.timeshift_multiple(X0, ..., device=True).dropna() -> sglm_cv.cv_glm_mult_params")}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        Ts = args.cpu_sample_T or 16_000
        v, v_sample, sec, sample, detail = cpu_reference_run(args, Ts, (0.0, 0.5, 1.0), 1, 1, 0)
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample, "sample_value": v_sample}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": step_ms, "higher_is_better": True,
                "scaling": "strong" if mode == "grid" else "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": config_dict(args, world, mode), "clocks": clocks, "e2e": e2e, "gpu_launches": launches,
                "roofline": roofline, "cpu_baseline": cpu,
                "best_params": res["best_params"], "best_score": float(res["best_score"])}
        if strong:
            line["strong_scaling"] = {"device_resident_step": device_timeline,
                                      "e2e_step_from_host_arrays": getattr(sglm_dist, "last_timeline", None),
                                      "unit": "ms per stage on rank 0 (CUDA events), last step of each leg"}
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
