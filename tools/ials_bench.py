"""Implicit-feedback ALS (iALS) at the ML-25M shape (162541 x 62423, dim 128): SvdEngine.ials_data / ials_sweep /
implicit_objective on the synthetic training split (synthetic.make_ratings at the ml25m shape, ~22.5 M ratings, merged into
~16.3 M distinct pairs of weight = count), tables drawn on the device with device_init_seed as tools/als_bench.py does.

Reports, in one JSON line (the GPU's name and power limit are read in the same run):
  - plan: ials_data from host arrays to a ready plan (merge, both CSRs, both row lists), host clock around a synchronise;
  - per sweep (CUDA events over warmed-up calls): G of each side (tfr_gram_rows), each half-sweep (its Gram included), the
    objective (two Grams + the observed pass), the whole sweep; the kernels' own times (torch.profiler, a run of its own);
  - the FP64 rate of each half-sweep from the FLOP count per side
        2 (sum_rows n (D (D + 1) / 2 + D) + rows (D^3 / 6 + D^2)) + 2 n_fixed D (D + 1) / 2,   D = dim,
    against the data sheet's 37 TFLOP/s for one B200 of an HGX B200 (a data-sheet fraction, not a measured peak);
  - HR / NDCG at 50 on the validation split (ratings >= 4 relevant, training pairs excluded) after each of 10 sweeps, for
    iALS and, on the same split and initialisation, for --solver als: context, not a claim.
Usage (GPU box): python tools/ials_bench.py [--out FILE] [--sweeps N] [--alpha A]"""
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import tf_recomm_b200  # noqa: E402,F401
from tf_recomm_b200 import config, synthetic  # noqa: E402
from tf_recomm_b200._lib import check  # noqa: E402
from tf_recomm_b200.engine import SvdEngine  # noqa: E402
from als_bench import kernel_label  # noqa: E402
from recommend_bench import FP64_DATASHEET, gpu_info, timed  # noqa: E402

K = 50


def flops(counts, n_fixed, dim):
    D = dim
    nz = counts[counts > 0]
    return (2.0 * (float(np.sum(nz, dtype=np.float64)) * (D * (D + 1) / 2 + D) + len(nz) * (D ** 3 / 6 + D ** 2))
            + 2.0 * n_fixed * D * (D + 1) / 2)


def calls(eng, data, alpha, reg):
    T = eng.t
    g_user = lambda: eng._gram(T["user_feat"], eng.U, data.user_gram, data.workspace)  # noqa: E731
    g_item = lambda: eng._gram(T["item_feat"], eng.I, data.item_gram, data.workspace)  # noqa: E731

    def user():
        g_item()
        eng._ials_half(data, alpha, reg, data.by_user, data.user_plan, (T["item_feat"], eng.I, data.item_gram),
                       (T["user_feat"], T["user_bias"]))

    def item():
        g_user()
        eng._ials_half(data, alpha, reg, data.by_item, data.item_plan, (T["user_feat"], eng.U, data.user_gram),
                       (T["item_feat"], T["item_bias"]))

    def objective():
        g_user()
        g_item()
        check(eng.L.tfr_ials_objective(
            T["user_feat"].data_ptr(), T["item_feat"].data_ptr(), eng.U, eng.I, eng.d, eng.feat_stride, eng.feat_stride,
            data.user_gram.data_ptr(), data.item_gram.data_ptr(), alpha, reg, data.by_user.indptr.data_ptr(),
            data.by_user.partner.data_ptr(), data.by_user.weight.data_ptr(), data.objective.data_ptr(),
            data.workspace.data_ptr(), data.workspace.numel(), eng._stream()))
    return dict(gram_user=g_user, gram_item=g_item, user_half=user, item_half=item, objective=objective)


def kernel_times(fns, reps=3):
    """Per-kernel device time (ms per call) from torch.profiler, each phase apart."""
    from torch.profiler import ProfilerActivity, profile
    out = {}
    for label in ("user_half", "item_half", "objective"):
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(reps):
                fns[label]()
            torch.cuda.synchronize()
        for ev in prof.key_averages():
            if "gram_" in ev.key or "ials_" in ev.key or "half_sweep_" in ev.key:
                name = kernel_label(ev.key)
                dt = getattr(ev, "device_time_total", None)
                if dt is None:
                    dt = ev.cuda_time_total
                out["%s.%s" % (label, name)] = dt / 1e3 / reps
    return out


def metrics(eng, vu, vi, vr, excl):
    m = eng.ranking_metrics(K, vu, vi, rates=vr, min_rating=4.0, exclude=excl)
    return dict(hr=m["hr"], ndcg=m["ndcg"], users=m["n_users"])


def main():
    out_path = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else None
    n_sweeps = int(sys.argv[sys.argv.index("--sweeps") + 1]) if "--sweeps" in sys.argv else 10
    alpha = float(sys.argv[sys.argv.index("--alpha") + 1]) if "--alpha" in sys.argv else 10.0
    name, power = gpu_info()
    reg = config.LAMBDA_REG
    res = dict(gpu=name, power_limit=power, alpha=alpha, reg=reg, fp64_datasheet_tflops=FP64_DATASHEET / 1e12)
    U, I, N = synthetic.SHAPES["ml25m"]
    d = 128
    users, items, rates = synthetic.make_ratings(U, I, N, seed=config.SEED)
    (tu, ti, tr), (vu, vi, vr) = synthetic.split(users, items, rates)
    del users, items, rates
    eng = SvdEngine(U, I, d, config.LEARNING_RATE, reg, device_init_seed=3)
    start = {n: eng.t[n].clone() for n in ("user_feat", "item_feat", "user_bias", "item_bias", "mu")}
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    data = eng.ials_data(tu, ti)
    torch.cuda.synchronize()
    res["plan_build_ms"] = (time.perf_counter() - t0) * 1e3
    cu = np.diff(data.by_user.indptr.cpu().numpy())
    ci = np.diff(data.by_item.indptr.cpu().numpy())
    res["shape"] = dict(users=U, items=I, dim=d, train_ratings=int(len(tu)), pairs=int(cu.sum()), val_ratings=int(len(vu)),
                        user_count_max=int(cu.max()), item_count_max=int(ci.max()))
    res["plan"] = dict(chunk=data.chunk, workspace_mb=data.workspace.numel() / 2 ** 20,
                       **{side + "_" + k: int(getattr(p, k).numel()) for side, p in (("user", data.user_plan),
                                                                                      ("item", data.item_plan))
                          for k in ("light", "heavy", "chunk_heavy")})
    excl = eng.pair_csr(tu, ti)
    # ---- 10 sweeps: implicit loss and HR / NDCG at 50 after each ----------------------------------------------------------
    curve = [dict(sweep=0, loss=eng.implicit_objective(data, alpha)["loss"])]
    for s in range(1, n_sweeps + 1):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        failed = eng.ials_sweep(data, alpha)
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) * 1e3
        curve.append(dict(sweep=s, sweep_ms=dt, loss=eng.implicit_objective(data, alpha)["loss"], failed=int(failed.item()),
                          **metrics(eng, vu, vi, vr, excl)))
        print(json.dumps(curve[-1]), file=sys.stderr)
    res["curve"] = curve
    # ---- phases (CUDA events, warmed up) -------------------------------------------------------------------------------
    fns = calls(eng, data, alpha, reg)
    ph = {k: timed(f, 20 if k.startswith("gram") or k == "objective" else 5)[0] for k, f in fns.items()}
    ph["sweep"] = timed(lambda: eng.ials_sweep(data, alpha), 3)[0]
    res["phases_ms"] = ph
    fl_u, fl_i = flops(cu, I, d), flops(ci, U, d)
    res["fp64"] = dict(user_flop=fl_u, item_flop=fl_i, user_tflops=fl_u / (ph["user_half"] * 1e-3) / 1e12,
                       item_tflops=fl_i / (ph["item_half"] * 1e-3) / 1e12,
                       user_datasheet_fraction=fl_u / (ph["user_half"] * 1e-3) / FP64_DATASHEET,
                       item_datasheet_fraction=fl_i / (ph["item_half"] * 1e-3) / FP64_DATASHEET,
                       sweep_datasheet_fraction=(fl_u + fl_i) / (ph["sweep"] * 1e-3) / FP64_DATASHEET)
    res["kernels_ms_per_call"] = kernel_times(fns)
    # ---- --solver als on the same split and initialisation, for context ----------------------------------------------------
    del data
    torch.cuda.empty_cache()
    for n, t in start.items():
        eng.t[n].copy_(t)
    adata = eng.als_data(tu, ti, tr)
    als_curve = []
    for s in range(1, n_sweeps + 1):
        eng.als_sweep(adata)
        als_curve.append(dict(sweep=s, **metrics(eng, vu, vi, vr, excl)))
        print(json.dumps(als_curve[-1]), file=sys.stderr)
    res["als_curve"] = als_curve
    line = json.dumps(res)
    print(line)
    if out_path:
        os.makedirs(os.path.dirname(out_path) or ".", exist_ok=True)
        with open(out_path, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
