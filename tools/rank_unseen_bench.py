"""Top-50 ranking of UNSEEN items at the ML-25M shape (162541 x 62423, dim 128, n_cand 64): rank_all_users without and
with the training pairs excluded (the exclusion set: synthetic.make_ratings at the ml25m shape, training split, ~22.5 M
pairs, deduplicated), the CSR build of that set, the ranking-metrics kernel over the [U, 50] ranking against the
validation split, the stage split of both sweeps (tfr_tune AP_STAGES, as tools/ap_stage_timing.py), and the ranking at
dim 15 at the ML-1M shape (every row through the exact float64 path).  CUDA events, warmed up.  Prints one JSON line.
Usage (GPU box): python tools/rank_unseen_bench.py [--reps N]"""
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import tf_recomm_b200  # noqa: E402,F401
from tf_recomm_b200 import _lib, config, synthetic  # noqa: E402
from tf_recomm_b200.engine import SvdEngine  # noqa: E402


def timed(fn, reps):
    """(mean ms over reps calls after one warm-up call, result of the last call)"""
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps, out


def split_pairs(shape):
    U, I, N = synthetic.SHAPES[shape]
    users, items, rates = synthetic.make_ratings(U, I, N, seed=config.SEED)
    return U, I, synthetic.split(users, items, rates)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    name, power = (x.strip() for x in q.stdout.strip().split(",")) if q.returncode == 0 else (torch.cuda.get_device_name(), "?")
    return name, power


def main():
    reps = int(sys.argv[sys.argv.index("--reps") + 1]) if "--reps" in sys.argv else 5
    k, n_cand = 50, 64
    name, power = gpu_info()
    res = dict(gpu=name, power_limit=power, k=k, n_cand=n_cand, reps=reps)

    U, I, ((tu, ti, _), (vu, vi, vr)) = split_pairs("ml25m")
    d = 128
    eng = SvdEngine(U, I, d, 1e-3, 0.05, device_init_seed=3)
    tu_d, ti_d = torch.from_numpy(tu).cuda(), torch.from_numpy(ti).cuda()
    keep = vr >= 4.0
    res["shape"] = dict(users=U, items=I, dim=d, train_pairs=int(len(tu)), val_relevant_pairs=int(keep.sum()))

    ms, out = timed(lambda: eng.rank_all_users(k=k, n_cand=n_cand), reps)
    res["unmasked_ms"], res["unmasked_n_uncertified"] = ms, out[2]
    ms, excl = timed(lambda: eng.pair_csr(tu_d, ti_d), reps)
    res["csr_build_ms"], res["excluded_pairs_distinct"] = ms, int(excl.items.numel())
    ms, out = timed(lambda: eng.rank_all_users(k=k, n_cand=n_cand, exclude=excl), reps)
    res["masked_rank_ms"], res["masked_n_uncertified"] = ms, out[2]
    res["masked_total_ms"] = res["csr_build_ms"] + res["masked_rank_ms"]
    res["masked_over_unmasked"] = res["masked_rank_ms"] / res["unmasked_ms"]
    idx = out[0]
    rel = eng.pair_csr(torch.from_numpy(vu[keep]).cuda(), torch.from_numpy(vi[keep]).cuda())
    ms, sums = timed(lambda: eng.ranking_sums(idx, rel), max(reps, 20))
    res["metrics_kernel_ms"] = ms
    s = sums.cpu().numpy()
    res["metrics_untrained_tables"] = dict(users=int(s[4]), hr=s[0] / s[4], recall=s[2] / s[4], ndcg=s[3] / s[4])

    # where the time goes: sweep + candidate buffers | + rescore | + exact rows (AP_STAGES bits 1 | 2 | 4)
    stages = {}
    for label, ex in (("unmasked", None), ("masked", excl)):
        for bits, what in ((1, "sweep"), (3, "sweep+rescore"), (7, "sweep+rescore+exact")):
            _lib.tune_set("AP_STAGES", bits)
            ms, _ = timed(lambda: eng.rank_all_users(k=k, n_cand=n_cand, exclude=ex), reps)
            stages["%s_%s_ms" % (label, what)] = ms
    _lib.tune_set("AP_STAGES", 7)
    # the same walk in the observed-pairs consumer, over the same (non-deduplicated) training pairs, against the plain
    # top-1 sweep: what a per-row CSR walk costs in the epilogue when it is not also feeding the candidate buffers
    indptr, it, rt = eng._csr_by_user(tu_d, ti_d, torch.ones_like(tu_d, dtype=torch.float32))
    row_se = torch.empty(U, dtype=torch.float64, device=eng.device)
    T = eng.t

    def obs_sweep():
        _lib.check(eng.L.tfr_allpairs_consume(T["user_feat"].data_ptr(), T["item_feat"].data_ptr(), T["user_bias"].data_ptr(),
                                              T["item_bias"].data_ptr(), T["mu"].data_ptr(), U, I, d, eng.feat_stride,
                                              eng.feat_stride, 0, 0, None, None, None, indptr.data_ptr(), it.data_ptr(),
                                              rt.data_ptr(), row_se.data_ptr(), None, 0, eng._stream()))
    stages["top1_sweep_ms"], _ = timed(lambda: eng.allpairs(use_tensor_cores=True), reps)
    stages["obs_walk_sweep_ms"], _ = timed(obs_sweep, reps)
    res["stages"] = stages
    del indptr, it, rt, row_se
    del eng, excl, rel, idx, out, tu_d, ti_d
    torch.cuda.empty_cache()

    U1, I1, ((tu1, ti1, _), _) = split_pairs("ml1m")
    eng1 = SvdEngine(U1, I1, 15, 1e-3, 0.05, device_init_seed=3)
    excl1 = eng1.pair_csr(tu1, ti1)
    ms, out = timed(lambda: eng1.rank_all_users(k=k, n_cand=n_cand, exclude=excl1), reps)
    res["ml1m_dim15"] = dict(users=U1, items=I1, dim=15, train_pairs=int(len(tu1)), masked_rank_ms=ms,
                             n_uncertified=out[2])
    print(json.dumps(res))


if __name__ == "__main__":
    main()
