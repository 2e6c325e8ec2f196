"""Top-50 of UNSEEN items for a batch of query users at the ML-25M shape (162541 x 62423, dim 128): SvdEngine.rank_users /
tfr_rank_users with the synthetic training split excluded (synthetic.make_ratings at the ml25m shape, ~22.5 M pairs; the
CSR is built once and timed on its own), for n = 1, 8, 64, 512, 4096, 32768 query users drawn with a fixed seed.

Per n: the device time of one call (CUDA events, device ids, warmed up), the scoring kernel alone against the whole call
(tfr_tune RANK_STAGES = 1 | 7), the achieved FP64 rate 2 n I d / time against the data sheet's 37 TFLOP/s for one B200 of
an HGX B200 (a data-sheet figure, not a measurement), the engine call end to end (host ids in, numpy out), and for
n <= 4096 get_ranking on the same users (which neither excludes nor ranks in float64).  In the same run: the masked
rank_all_users sweep over every user, and the n from which it is the cheaper way.  Prints one JSON line.
Usage (GPU box): python tools/recommend_bench.py [--out FILE]"""
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import tf_recomm_b200  # noqa: E402,F401
from tf_recomm_b200 import _lib, config, synthetic  # noqa: E402
from tf_recomm_b200.engine import SvdEngine  # noqa: E402

FP64_DATASHEET = 37e12   # FLOP/s, one GPU of an HGX B200 (the data sheet prints 296 TFLOP/s for eight)
NS = (1, 8, 64, 512, 4096, 32768)


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


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    name, power = (x.strip() for x in q.stdout.strip().split(",")) if q.returncode == 0 else (torch.cuda.get_device_name(), "?")
    return name, power


def main():
    out_path = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else None
    k, d = 50, 128
    name, power = gpu_info()
    res = dict(gpu=name, power_limit=power, k=k, fp64_datasheet_tflops=FP64_DATASHEET / 1e12)
    U, I, N = synthetic.SHAPES["ml25m"]
    users, items, rates = synthetic.make_ratings(U, I, N, seed=config.SEED)
    (tu, ti, _), _ = synthetic.split(users, items, rates)
    del users, items, rates
    eng = SvdEngine(U, I, d, 1e-3, 0.05, device_init_seed=3)
    tu_d, ti_d = torch.from_numpy(tu).cuda(), torch.from_numpy(ti).cuda()
    res["shape"] = dict(users=U, items=I, dim=d, train_pairs=int(len(tu)))
    res["csr_build_ms"], excl = timed(lambda: eng.pair_csr(tu_d, ti_d), 5)
    res["excluded_pairs_distinct"] = int(excl.items.numel())
    res["rank_all_users_masked_ms"], _ = timed(lambda: eng.rank_all_users(k=k, exclude=excl), 5)
    T = eng.t
    rng = np.random.default_rng(2024)
    rows = []
    for n in NS:
        q = rng.integers(0, U, n).astype(np.int32)
        q_dev = torch.from_numpy(q).cuda()
        idx = torch.empty(n, k, dtype=torch.int32, device=eng.device)
        val = torch.empty(n, k, dtype=torch.float64, device=eng.device)
        nbytes = eng.L.tfr_rank_users_workspace_bytes(n, I, k)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=eng.device)

        def call():
            _lib.check(eng.L.tfr_rank_users(T["user_feat"].data_ptr(), T["item_feat"].data_ptr(), T["user_bias"].data_ptr(),
                                            T["item_bias"].data_ptr(), T["mu"].data_ptr(), U, I, d, eng.feat_stride,
                                            eng.feat_stride, eng.flags, q_dev.data_ptr(), n, k, excl.indptr.data_ptr(),
                                            excl.items.data_ptr(), val.data_ptr(), idx.data_ptr(), ws.data_ptr(), nbytes,
                                            eng._stream()))
        reps = max(3, min(200, 200000 // n))
        r = dict(n=n, reps=reps, workspace_mb=nbytes / 2**20)
        _lib.tune_set("RANK_STAGES", 1)
        r["score_only_ms"], _ = timed(call, reps)
        _lib.tune_set("RANK_STAGES", 3)
        r["score_select_ms"], _ = timed(call, reps)
        _lib.tune_set("RANK_STAGES", 7)
        r["device_ms"], _ = timed(call, reps)
        r["us_per_query"] = 1e3 * r["device_ms"] / n
        flop = 2.0 * n * I * d
        r["fp64_tflops"] = flop / (r["device_ms"] * 1e-3) / 1e12
        r["fp64_fraction_of_datasheet"] = r["fp64_tflops"] * 1e12 / FP64_DATASHEET
        r["score_only_fp64_fraction_of_datasheet"] = flop / (r["score_only_ms"] * 1e-3) / FP64_DATASHEET
        eng.rank_users(q, k=k, exclude=excl)   # warm-up: the engine's cached workspace for (n, k)
        torch.cuda.synchronize()
        e2e = []
        for _ in range(max(3, min(20, reps))):
            t0 = time.perf_counter()
            a, b = eng.rank_users(q, k=k, exclude=excl)
            a.cpu().numpy(), b.cpu().numpy()
            e2e.append((time.perf_counter() - t0) * 1e3)
        r["engine_e2e_ms_median"] = float(np.median(e2e))
        del a, b
        eng._stage.pop(("rank_users_ws", n, k), None)
        if n <= 4096:
            r["get_ranking_ms"], _ = timed(lambda: eng.get_ranking(q, k=k), 3 if n >= 512 else 10)
        rows.append(r)
        print(json.dumps(r), file=sys.stderr)
        del ws, idx, val, q_dev
        torch.cuda.empty_cache()
    res["queries"] = rows
    # where the full sweep becomes cheaper: the n at which the per-call time, linear between the two measured sizes that
    # bracket the sweep's time (or extrapolated from the last two), reaches it
    sweep = res["rank_all_users_masked_ms"]
    ns, ts = [r["n"] for r in rows], [r["device_ms"] for r in rows]
    j = next((j for j in range(1, len(ns)) if ts[j] >= sweep), len(ns) - 1)
    slope = (ts[j] - ts[j - 1]) / (ns[j] - ns[j - 1])
    res["crossover_n"] = int(round(ns[j - 1] + (sweep - ts[j - 1]) / slope)) if slope > 0 else None
    res["crossover_measured_bracket"] = ts[-1] >= sweep
    line = json.dumps(res)
    print(line)
    if out_path:
        os.makedirs(os.path.dirname(out_path) or ".", exist_ok=True)
        with open(out_path, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
