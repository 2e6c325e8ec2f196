"""Similar items and users (SvdEngine.similar_items / similar_users, tfr_similar_rows) next to rank_users at the ML-25M
shape: 162,541 users x 62,423 items, dim 128, k = 50, tables drawn on the device (Adam layout, stride 3d).

  * similar_items for n = 1, 64, 4,096 and all 62,423 items; similar_users for n = 1, 64, 4,096;
  * each next to rank_users (nothing excluded) at the same n, the two calls alternated within one run;
  * CUDA events around `--reps` calls after `--warmup` calls of every shape; the mean per call is reported.
rank_users scores n x 62,423 pairs, similar_items n x 62,423 and similar_users n x 162,541: the same float64 FMA count
per pair, plus one DMUL and one DDIV per pair and the norm pass over the candidate table.  The card's name and power
limit are read in the same run.  Writes one JSON file (--out).
Usage (GPU box): python tools/similar_bench.py --out F.json"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import tf_recomm_b200  # noqa: E402,F401
from tf_recomm_b200.engine import SvdEngine  # noqa: E402

U, I, D, K = 162541, 62423, 128, 50


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    name, power = (x.strip() for x in q.stdout.strip().split(",")) if q.returncode == 0 else (torch.cuda.get_device_name(), "?")
    return name, power


def timed(fns, reps, warmup):
    """{name: mean ms per call}; the calls of fns alternate, each timed by its own pair of events per call."""
    for _ in range(warmup):
        for fn in fns.values():
            fn()
    torch.cuda.synchronize()
    tot = {n: 0.0 for n in fns}
    for _ in range(reps):
        for n, fn in fns.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            tot[n] += a.elapsed_time(b)
    return {n: t / reps for n, t in tot.items()}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a GPU"
    name, power = gpu_info()
    eng = SvdEngine(U, I, D, 1e-3, 0.05, device_init_seed=7)
    rng = np.random.default_rng(0)
    rows = []
    cases = [("items", n) for n in (1, 64, 4096, I)] + [("users", n) for n in (1, 64, 4096)]
    for side, n in cases:
        qs = torch.from_numpy((np.arange(I) if n == I else rng.integers(0, I if side == "items" else U, n))
                              .astype(np.int32)).cuda()
        qu = torch.from_numpy(rng.integers(0, U, n).astype(np.int32)).cuda()
        sim = (lambda: eng.similar_items(qs, K)) if side == "items" else (lambda: eng.similar_users(qs, K))
        fns = {"similar_" + side: sim, "rank_users": lambda: eng.rank_users(qu, K)}
        ms = timed(fns, max(1, args.reps if n < I else 2), args.warmup if n < I else 1)
        cand = I if side == "items" else U
        rows.append(dict(call="similar_" + side, n=n, k=K, candidates=cand, ms=ms["similar_" + side],
                         rank_users_ms=ms["rank_users"], ratio=ms["similar_" + side] / ms["rank_users"],
                         pairs_per_s=n * cand / (ms["similar_" + side] * 1e-3),
                         rank_users_pairs_per_s=n * I / (ms["rank_users"] * 1e-3)))
        print(json.dumps(rows[-1]), flush=True)
        del qs, qu
        eng._stage.clear()   # the cached workspaces of this shape
        torch.cuda.empty_cache()
    out = dict(gpu=name, power_limit=power, shape=dict(users=U, items=I, dim=D, k=K, layout="adam (stride 3d)"),
               timing="CUDA events per call, calls alternated, mean over warmed-up calls", rows=rows)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
