"""Fold-in of users at the ML-25M shape (162541 x 62423, dim 128): tfr_fold_in_users / SvdEngine.fold_in on the synthetic
training split's ratings (synthetic.make_ratings at the ml25m shape, ~22.5 M ratings), item tables drawn on the device with
device_init_seed as tools/recommend_bench.py does.

Per n (one median-count user, the heaviest user alone, 64 and 4096 users drawn with a fixed seed, every user = one user
half-sweep of ALS): the device time of one call (CUDA events over warmed-up calls, CSR on the device), and the achieved FP64
rate from the FLOP count 2 (sum_u n_u (D (D + 1) / 2 + D) + n (D^3 / 6 + D^2)), D = dim + 1 (Gram + right-hand side, then
Cholesky + the two substitutions), against the data sheet's 37 TFLOP/s for one B200 of an HGX B200 (a data-sheet figure,
not a measurement).  Also: the serving latency of SvdEngine.fold_in + rank_folded(k = 50) for one new user with 100
ratings (host arrays in, numpy out), and the whole-population call at the ML-1M README shape (dim 15).  The GPU's name and
power limit are read in the same run.  Prints one JSON line.
Usage (GPU box): python tools/fold_in_bench.py [--out FILE]"""
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
from tf_recomm_b200 import _lib, config, synthetic  # noqa: E402
from tf_recomm_b200.engine import SvdEngine  # noqa: E402
from recommend_bench import FP64_DATASHEET, gpu_info, timed  # noqa: E402

REG = 0.05


def flops(counts, dim):
    D = dim + 1
    return 2.0 * (float(np.sum(counts, dtype=np.float64)) * (D * (D + 1) / 2 + D) + len(counts) * (D ** 3 / 6 + D ** 2))


def measure(eng, tu, ti, tr, users, label):
    """Fold-in of the given users from their training ratings: CSR built once, then the C call timed alone."""
    order = np.argsort(tu, kind="stable")
    starts = np.searchsorted(tu[order], np.arange(eng.U + 1))
    sel = np.concatenate([order[starts[u]:starts[u + 1]] for u in users]) if len(users) < eng.U else order
    row_of = np.empty(eng.U, np.int64)
    row_of[users] = np.arange(len(users))
    f = eng.fold_in(row_of[tu[sel]], ti[sel], tr[sel], n=len(users), reg=REG)
    counts = (f.ratings.indptr[1:] - f.ratings.indptr[:-1]).cpu().numpy()
    indptr, items = f.ratings.indptr, f.ratings.items
    rates = torch.from_numpy(tr[sel]).cuda()   # (timing only: the rates' order does not change the work)
    n = len(users)
    T = eng.t

    def call():
        _lib.check(eng.L.tfr_fold_in_users(T["item_feat"].data_ptr(), T["item_bias"].data_ptr(), T["mu"].data_ptr(), eng.I,
                                           eng.d, eng.feat_stride, eng.flags, REG, indptr.data_ptr(), items.data_ptr(),
                                           rates.data_ptr(), n, f.feat.data_ptr(), f.bias.data_ptr(), f.info.data_ptr(),
                                           eng._stream()))
    reps = max(3, min(200, 20000 // n))
    ms, _ = timed(call, reps)
    fl = flops(counts, eng.d)
    r = dict(case=label, n=n, ratings=int(counts.sum()), max_ratings=int(counts.max()), reps=reps, device_ms=ms,
             flop=fl, fp64_tflops=fl / (ms * 1e-3) / 1e12, fp64_fraction_of_datasheet=fl / (ms * 1e-3) / FP64_DATASHEET,
             info_nonzero=int((f.info != 0).sum()))
    print(json.dumps(r), file=sys.stderr)
    return r


def main():
    out_path = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else None
    name, power = gpu_info()
    res = dict(gpu=name, power_limit=power, reg=REG, fp64_datasheet_tflops=FP64_DATASHEET / 1e12)
    U, I, N = synthetic.SHAPES["ml25m"]
    d = 128
    users, items, rates = synthetic.make_ratings(U, I, N, seed=config.SEED)
    (tu, ti, tr), _ = synthetic.split(users, items, rates)
    del users, items, rates
    eng = SvdEngine(U, I, d, 1e-3, REG, device_init_seed=3)
    counts = np.bincount(tu, minlength=U)
    res["shape"] = dict(users=U, items=I, dim=d, train_ratings=int(len(tu)), count_median=float(np.median(counts)),
                        count_p99=float(np.percentile(counts, 99)), count_max=int(counts.max()))
    t0 = time.perf_counter()
    eng.fold_in(tu, ti, tr, n=U, reg=REG)
    torch.cuda.synchronize()
    res["engine_fold_in_all_users_host_arrays_ms"] = (time.perf_counter() - t0) * 1e3
    rng = np.random.default_rng(2024)
    median_user = int(np.nonzero(counts == int(np.median(counts)))[0][0])
    rows = [measure(eng, tu, ti, tr, np.array([median_user]), "1 median-count user"),
            measure(eng, tu, ti, tr, np.array([int(counts.argmax())]), "1 heaviest user"),
            measure(eng, tu, ti, tr, np.sort(rng.choice(U, 64, replace=False)), "64 users"),
            measure(eng, tu, ti, tr, np.sort(rng.choice(U, 4096, replace=False)), "4096 users"),
            measure(eng, tu, ti, tr, np.arange(U), "every user")]
    res["calls"] = rows
    # serving: one new user with 100 ratings, host arrays in, numpy out
    it = rng.choice(I, 100, replace=False).astype(np.int32)
    rt = rng.integers(1, 6, 100).astype(np.float32)
    zeros = np.zeros(100, np.int64)

    def serve():
        f = eng.fold_in(zeros, it, rt, reg=REG)
        a, b = eng.rank_folded(f, k=50)
        return a.cpu().numpy(), b.cpu().numpy()
    for _ in range(3):
        serve()
    e2e = []
    for _ in range(30):
        t0 = time.perf_counter()
        serve()
        e2e.append((time.perf_counter() - t0) * 1e3)
    res["serving_fold_in_plus_top50_one_user_100_ratings_ms_median"] = float(np.median(e2e))
    del eng
    torch.cuda.empty_cache()
    # README shape: ML-1M, dim 15, every user
    U1, I1, N1 = synthetic.SHAPES["ml1m"]
    u1, i1, r1 = synthetic.make_ratings(U1, I1, N1, seed=config.SEED)
    (tu1, ti1, tr1), _ = synthetic.split(u1, i1, r1)
    eng1 = SvdEngine(U1, I1, 15, 1e-3, REG, device_init_seed=3)
    res["readme_shape"] = measure(eng1, tu1, ti1, tr1, np.arange(U1), "every user, ML-1M, dim 15")
    line = json.dumps(res)
    print(line)
    if out_path:
        os.makedirs(os.path.dirname(out_path) or ".", exist_ok=True)
        with open(out_path, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
