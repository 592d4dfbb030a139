"""Row-sharded log-link GLM grids: the staged weighted tcgen05 Gram summed over row slices against the one-shot Gram,
the batched solver with a single-process `comm` against comm=None, and (2+ GPUs) sglm_dist.cv_grid_strong with
Poisson / Gamma / Tweedie sets against the one-GPU grid."""
import ctypes
import os
import socket
import sys

import numpy as np
import pytest

from conftest import PKG, ROOT, coef_rel_err

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
if not torch.cuda.is_available():
    pytest.skip("needs a CUDA device", allow_module_level=True)

import synth_data  # noqa: E402
import _engine as eng  # noqa: E402
import _sglm_native as nat  # noqa: E402
from oracle import sglm_oracle as orc  # noqa: E402


def _design(T, P, seed):
    shifts = [0] + [s for s in range(-3, 5) if s != 0]
    Xd = orc.timeshift_multiple(synth_data.synth_base(T, P, seed), shift_amt_list=shifts)
    Xd = Xd[~np.isnan(Xd).any(axis=1)]
    return Xd, synth_data.synth_kernels(P, shifts, seed)


def _staged_gram(Xd, Yd, rs, max_planes, cuts):
    """The weighted Gram from row slices [cuts[k], cuts[k+1]) through the staged ABI, the int64 partials added here."""
    n_y, (T, C) = Yd.shape[1], Xd.shape
    n_aug = C + n_y + 1
    ldg = eng._round_up(n_aug, 8)
    sl = list(zip(cuts[:-1], cuts[1:]))
    cm, ls = [], []
    for a, b in sl:
        colmax = torch.empty(n_aug, dtype=torch.int64, device="cuda")
        lsb = torch.empty(n_aug, dtype=torch.int32, device="cuda")
        Xs, Ys, rss = Xd[a:b], Yd[a:b], rs[a:b]
        assert nat.lib().sglm_gram_tc_colstats_scaled_f64(eng.ptr(Xs), C, eng.ptr(Ys), n_y, n_y, b - a, C,
                                                          eng.ptr(rss) if b > a else None, eng.ptr(colmax), eng.ptr(lsb),
                                                          nat.stream_ptr()) == 0
        cm.append(colmax)
        ls.append(lsb)
    colmax = torch.stack(cm).max(dim=0).values.contiguous()
    colS = torch.stack(ls).min(dim=0).values.contiguous()
    colE = torch.empty(n_aug, dtype=torch.int32, device="cuda")
    flag = torch.empty(1, dtype=torch.int32, device="cuda")
    eng.call("sglm_gram_tc_exponents", eng.ptr(colmax), n_aug, max_planes, eng.ptr(colE), eng.ptr(colS), eng.ptr(flag),
             nat.stream_ptr())
    colS_h = np.ascontiguousarray(colS.cpu().numpy(), dtype=np.int32)
    member = np.ones((1, 1), dtype=np.int32)
    total, keep = None, None
    for a, b in sl:
        n = b - a
        rows = torch.full((max(eng._round_up(n, 128), 128),), -1, dtype=torch.int64, device="cuda")
        rows[:n] = torch.arange(n, dtype=torch.int64, device="cuda")
        sizes = np.array([n], dtype=np.int64)
        cp, sp = colS_h.ctypes.data_as(ctypes.c_void_p), sizes.ctypes.data_as(ctypes.c_void_p)
        wsb = nat.lib().sglm_gram_tc_cells_workspace_bytes(n_aug, cp, 1, sp, 1)
        ob, nb = ctypes.c_uint64(0), ctypes.c_uint64(0)
        assert nat.lib().sglm_gram_tc_cells_sgout(n_aug, cp, 1, sp, 1, ctypes.byref(ob), ctypes.byref(nb)) == 0
        raw = torch.empty(wsb + 1024, dtype=torch.uint8, device="cuda")
        off = (-raw.data_ptr()) % 1024
        ws = ctypes.c_void_p(raw.data_ptr() + off)
        Xs, Ys, rss = Xd[a:b], Yd[a:b], rs[a:b]
        eng.call("sglm_gram_tc_scaled_partial_f64", eng.ptr(Xs), C, eng.ptr(Ys), n_y, n_y, n, C,
                 eng.ptr(rss) if n else None, eng.ptr(colE), eng.ptr(colS), cp, 1, sp, eng.ptr(rows), 1,
                 member.ctypes.data_as(ctypes.c_void_p), ws, wsb, nat.stream_ptr())
        sg = raw[off + ob.value: off + ob.value + nb.value].view(torch.int64)
        total = sg.clone() if total is None else total + sg
        keep = (raw, off, ob.value, nb.value, ws, wsb, cp, sp, sizes)
    raw, off, o, nbytes, ws, wsb, cp, sp, _ = keep
    raw[off + o: off + o + nbytes].view(torch.int64).copy_(total)
    G = eng._zeros((1, n_aug, ldg))
    eng.call("sglm_gram_tc_cells_combine_f64", C, n_y, eng.ptr(colE), eng.ptr(colS), cp, 1, sp, 1, eng.ptr(G), ldg, ws,
             wsb, nat.stream_ptr())
    return G


@pytest.mark.parametrize("max_planes", [eng.POISSON_TC_PLANES, 2, 8])
def test_staged_weighted_gram_over_row_slices_is_bit_identical(max_planes):
    """Ragged slices, an empty slice, 0/1 and real columns; max_planes below what the real columns need (2, 4) and
    at the maximum (8)."""
    Xd, _ = _design(2900, 4, 7)
    T = Xd.shape[0]
    X = torch.from_numpy(Xd).cuda()
    rng = np.random.default_rng(7)
    Y = torch.from_numpy(rng.gamma(2.0, 1.0, (T, 1))).cuda()
    rs = torch.from_numpy(np.sqrt(rng.gamma(1.5, 1.0, T))).cuda()
    assert any(np.all((Xd[:, c] == 0) | (Xd[:, c] == 1)) for c in range(Xd.shape[1]))
    one = eng.suffstats_tc_scaled(X, Y, rs, max_planes)
    for cuts in ([0, T], [0, 1, 700, 700, 2051, T], [0, 129, 128 * 7, T - 3, T]):
        G = _staged_gram(X, Y, rs, max_planes, cuts)
        assert torch.equal(G, one), (cuts, float((G - one).abs().max()))


class _OneRank:
    """comm of a single process: nothing to exchange, the partials pass through the fixed-order sum."""

    def all_reduce(self, t, op):
        assert op in ("max", "min", "sum")

    def combine(self, t):
        return eng.reduce_parts(t.reshape(-1).contiguous(), 1).reshape(t.shape)


def _grid_inputs(power, seed=5):
    Xd, beta = _design(3000, 4, seed)
    T = Xd.shape[0]
    if power == 1:
        y = synth_data.synth_response(Xd, beta, seed, poisson=True)
    else:
        y = synth_data.synth_response_tweedie(Xd, beta, seed, power)
    folds = synth_data.synth_folds(T, 3, seed, group=100)
    X = torch.from_numpy(Xd).cuda()
    yd = torch.from_numpy(np.ascontiguousarray(y, dtype=np.float64)).cuda()
    Yd = torch.stack([yd, eng.roll_vector(yd, 5)], dim=1).contiguous()
    te = [eng.index_counts(b, T) for _, b in folds]
    tr = [eng.index_counts(a, T) for a, _ in folds]
    RW = torch.stack(tr + te).contiguous()
    F = len(folds)
    models, ycol, rw_a, rw_b = [], [], [], []
    for alpha, yc, fi in ((1e-3, 0, True), (1e-1, 1, True), (1e-2, 0, False)):
        for f in range(F):
            models.append(eng.PoissonModel(alpha, fi, rw=f, ycol=yc))
            ycol.append(yc); rw_a.append(f); rw_b.append(F + f)
        models.append(eng.PoissonModel(alpha, fi, rw=-1, ycol=0))
        ycol.append(0); rw_a.append(-1); rw_b.append(-2)
    return X, Yd, RW, models, ycol, rw_a, rw_b


@pytest.mark.parametrize("use_tc", [True, False])
@pytest.mark.parametrize("power", [1.0, 1.5, 2.0, 3.0])
def test_single_rank_comm_is_bit_identical(power, use_tc):
    X, Yd, RW, models, ycol, rw_a, rw_b = _grid_inputs(power)
    old = eng.POISSON_TC
    eng.POISSON_TC = use_tc
    try:
        W0, b0, it0, st0 = eng.tweedie_grid_batched(X, Yd, models, RW, power)
        tc0 = eng.last_poisson_batch[0]["tensor_core_hessian"]
        W1, b1, it1, st1 = eng.tweedie_grid_batched(X, Yd, models, RW, power, comm=_OneRank())
        tc1 = eng.last_poisson_batch[0]["tensor_core_hessian"]
    finally:
        eng.POISSON_TC = old
    assert tc0 == tc1 == use_tc
    assert set(np.unique(st0)) <= {1, 2}
    assert torch.equal(W0, W1) and torch.equal(b0, b1)
    assert np.array_equal(it0, it1) and np.array_equal(st0, st1)
    s0 = eng.tweedie_scores_batched(X, Yd, W0, b0, ycol, rw_a, rw_b, RW, power)
    s1 = eng.tweedie_scores_batched(X, Yd, W0, b0, ycol, rw_a, rw_b, RW, power, comm=_OneRank())
    assert np.array_equal(s0, s1)


# --------------------------------------------------------------------------- #
# 2+ GPUs: sglm_dist.cv_grid_strong over NCCL
# --------------------------------------------------------------------------- #
N_GPUS = torch.cuda.device_count()
SHIFTS = [0] + [s for s in range(-3, 5) if s != 0]
GRID = ([dict(alpha=a, l1_ratio=0.5, max_iter=1000) for a in (1e-3, 1e-2)] +
        [dict(model_name="Poisson", alpha=a, max_iter=100) for a in (1e-3, 1e-1)] +
        [dict(model_name="Gamma", alpha=1e-2), dict(model_name="Tweedie", power=1.5, alpha=1e-2),
         dict(model_name="Poisson", alpha=1e-2, roll=11)])


def _inputs():
    X0 = synth_data.synth_base(6000, 4, 21)
    d = orc.timeshift_multiple(X0, shift_amt_list=SHIFTS)[4:-3]
    assert not np.isnan(d).any()
    y = synth_data.synth_response_tweedie(d, synth_data.synth_kernels(4, SHIFTS, 21), 21, 2.0)       # y > 0: every family
    folds = synth_data.synth_folds(d.shape[0], 4, 21, group=150)
    return X0, d, y, folds


def _record(res):
    """Everything a result dict holds, as bytes: two ranks' records compare equal only when every bit does."""
    out = [repr(res["best_params"]), np.float64(res["best_score"]).tobytes()]
    for r in res["full_cv_results"]:
        out.append(repr(r["glm_kwargs"]))
        for k in ("cv_coefs", "cv_intercepts", "cv_scores_train", "cv_scores_test", "cv_mean_score_train",
                  "cv_mean_score", "cv_std_score", "cv_R2_score", "cv_mse_score"):
            out.append(np.asarray(r[k], dtype=np.float64).tobytes())
        out.append(np.asarray(r["model"].coef_).tobytes() + np.float64(r["model"].intercept_).tobytes())
    return out


def _worker(rank, world, port, backend, ret):
    for p in (ROOT, PKG):
        if p not in sys.path:
            sys.path.insert(0, p)
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    if backend == "nccl":
        torch.cuda.set_device(rank)
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    else:                                       # gloo: every rank on GPU 0, the collectives on its CUDA tensors
        torch.cuda.set_device(0)
        dist.init_process_group("gloo", rank=rank, world_size=world)
    import sglm_cv
    import sglm_dist
    import sglm_pp
    X0, d, y, folds = _inputs()
    mine = [None] * world
    res = sglm_dist.cv_grid_strong(X0 if rank == 0 else None, SHIFTS, y if rank == 0 else None,
                                   folds if rank == 0 else None, "Gaussian", [dict(g) for g in GRID], score_method="r2")
    dist.all_gather_object(mine, _record(res))
    report = {"ranks_identical": all(m == mine[0] for m in mine)}
    # a negative y for Poisson: the one-GPU exception on EVERY rank, no rank left waiting in a collective
    y_bad = y.copy()
    y_bad[len(y) // 3] = -1.0
    try:
        sglm_dist.cv_grid_strong(X0 if rank == 0 else None, SHIFTS, y_bad if rank == 0 else None,
                                 folds if rank == 0 else None, "Gaussian", [dict(g) for g in GRID[2:4]])
        report["bad_y"] = "no exception"
    except ValueError as e:
        report["bad_y"] = str(e)
    if rank == 0:
        os.environ["SGLM_GRAM"] = "tc"          # the one-GPU Gaussian statistics on the same (exact) path
        try:
            lazy = sglm_pp.timeshift_multiple(torch.from_numpy(X0).cuda(), shift_amt_list=SHIFTS, device=True).dropna()
            one = sglm_cv.cv_glm_mult_params(lazy, y, folds, "Gaussian", [dict(g) for g in GRID], score_method="r2")
        finally:
            os.environ.pop("SGLM_GRAM", None)
        report["best_params"] = (res["best_params"], one["best_params"])
        worst = dict(coef=0.0, icpt=0.0, score=0.0, gauss_score=0.0, iters=0, gauss_coef_equal=True)
        for a, b, g in zip(res["full_cv_results"], one["full_cv_results"], GRID):
            if g.get("model_name", "Gaussian") == "Gaussian":
                worst["gauss_coef_equal"] &= bool(np.array_equal(a["cv_coefs"], b["cv_coefs"]) and
                                                  np.array_equal(a["cv_intercepts"], b["cv_intercepts"]) and
                                                  np.array_equal(a["model"].coef_, b["model"].coef_) and
                                                  a["model"].intercept_ == b["model"].intercept_)
                for k in ("cv_scores_train", "cv_scores_test", "cv_R2_score", "cv_mse_score"):
                    worst["gauss_score"] = max(worst["gauss_score"], float(np.max(np.abs(np.subtract(a[k], b[k])))))
                continue
            for j in range(a["cv_coefs"].shape[1]):
                worst["coef"] = max(worst["coef"], coef_rel_err(a["cv_coefs"][:, j], b["cv_coefs"][:, j]))
            worst["coef"] = max(worst["coef"], coef_rel_err(a["model"].coef_, b["model"].coef_))
            worst["icpt"] = max(worst["icpt"], float(np.max(np.abs(a["cv_intercepts"] - b["cv_intercepts"]))),
                                abs(a["model"].intercept_ - b["model"].intercept_))
            for k in ("cv_scores_train", "cv_scores_test", "cv_mean_score", "cv_R2_score", "cv_mse_score"):
                worst["score"] = max(worst["score"], float(np.max(np.abs(np.subtract(a[k], b[k])))))
            worst["iters"] = max(worst["iters"], int(np.max(np.abs(a["_fit_info"]["n_iter"].astype(np.int64) -
                                                                   b["_fit_info"]["n_iter"].astype(np.int64)))))
        report["worst"] = worst
    ret[rank] = report
    dist.barrier()
    dist.destroy_process_group()


def _spawn(world, backend, timeout=600):
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    mgr = mp.Manager()
    try:
        ret = mgr.dict()
        ctx = mp.start_processes(_worker, args=(world, port, backend, ret), nprocs=world, join=False, start_method="spawn")
        import time
        deadline = time.monotonic() + timeout
        try:
            while not ctx.join(timeout=5):
                if time.monotonic() > deadline:
                    raise TimeoutError(f"cv_grid_strong over {world} GPUs did not finish in {timeout} s")
        finally:
            for p in ctx.processes:
                if p.is_alive():
                    p.terminate()
                p.join()
        return dict(ret)
    finally:
        mgr.shutdown()


@pytest.mark.parametrize("world,backend", [(2, "nccl"), (4, "nccl"), (2, "gloo")])
def test_strong_grid_log_link_families(world, backend):
    """NCCL: one GPU per rank.  gloo: the ranks share GPU 0 — the row sharding and the lock step on one device."""
    if backend == "nccl" and N_GPUS < world:
        pytest.skip(f"needs {world} GPUs")
    out = _spawn(world, backend)
    assert sorted(out) == list(range(world))
    bad = "Some value(s) of y are out of the valid range of the loss 'HalfPoissonLoss'."
    for r in range(world):
        assert out[r]["ranks_identical"], r
        assert out[r]["bad_y"] == bad, (r, out[r]["bad_y"])
    got, want = out[0]["best_params"]
    assert got == want
    w = out[0]["worst"]
    print(f"world {world} ({backend}): {w}")
    assert w["gauss_coef_equal"]
    # Gaussian scores are quadratic forms whose row split follows the models a rank scores at once (last bits)
    assert w["gauss_score"] <= 1e-12, w
    # log link: the fp64 gradient sums are re-associated over the ranks; the iterates reach the same fixed point
    # (observed on a B200, 2 ranks: 1e-14 relative in the coefficients, 3e-15 in the scores, equal n_iter)
    assert w["coef"] <= 1e-11 and w["icpt"] <= 1e-11 and w["score"] <= 1e-12 and w["iters"] <= 1, w
