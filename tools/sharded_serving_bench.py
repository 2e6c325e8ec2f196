"""Serving from row-sharded tables (ShardedSvdEngine.rank_users / fold_in / rank_folded), timed with CUDA events.

Under torchrun (NCCL, one process per GPU, WORLD_SIZE >= 2), at the BASELINE configs[4] shape (100M users x 10M items,
dim 128; bench_sharded.sharded_config, tables drawn on the device as bench_sharded draws them):
  * an in-run parity check first, at tables scaled down 1000x: rank 0 re-assembles the tables and compares rank_users
    (with training pairs excluded) and fold_in + rank_folded with SvdEngine, ids and bits;
  * rank_users for n = 1, 64 and 4096 query users, k = 50, nothing excluded (configs[4] has no fixed training set);
  * fold_in + rank_folded of 1 and 4096 new users with 100 synthetic ratings each;
  * per rank, the split of every call: local ranking (tfr_rank_users on the item shard), merge (tfr_shard_topk_merge),
    collectives (all-reduce of the gathered rows, all-gather of the lists) and the rest (row gather, exclusion lists,
    fold-in solve).
Without torchrun (world 1): the ML-25M shape (162541 x 62423, dim 128), ShardedSvdEngine.rank_users at world 1 next to
SvdEngine.rank_users on the same tables (calls alternated), bit equality checked -- what the gather and merge layer
costs.  Every call is warmed up; the mean over the timed calls is reported.  The card's name and power limit are read in
the same run.  Writes one JSON file (--out).
Usage (GPU box): python tools/sharded_serving_bench.py --out F.json
                 torchrun --nproc-per-node N tools/sharded_serving_bench.py --out F.json"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench_sharded  # noqa: E402
import tf_recomm_b200  # noqa: E402,F401
from tf_recomm_b200 import sharding  # noqa: E402
from tf_recomm_b200.engine import SvdEngine  # noqa: E402
from tf_recomm_b200.sharded import ShardedSvdEngine  # noqa: E402

K, N_RATINGS = 50, 100
LR, REG = bench_sharded.LR, bench_sharded.REG


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    name, power = (x.strip() for x in q.stdout.strip().split(",")) if q.returncode == 0 else (torch.cuda.get_device_name(), "?")
    return name, power


class Phases:
    """CUDA events around the phases of one call, on the current stream (a collective's work joins it before return)."""

    def __init__(self):
        self.marks = []

    def mark(self, name):
        ev = torch.cuda.Event(enable_timing=True)
        ev.record()
        self.marks.append((name, ev))

    def split(self):
        torch.cuda.synchronize()
        out = {}
        for (_, a), (name, b) in zip(self.marks, self.marks[1:]):
            out[name] = out.get(name, 0.0) + a.elapsed_time(b)
        return out


def rank_users_phased(eng, q, k, ph):
    """ShardedSvdEngine.rank_users (nothing excluded) with its phases marked."""
    n, d = q.numel(), eng.d
    ph.mark("start")
    table = eng.serve_gather(q)
    ph.mark("other")
    eng._all_reduce(table)
    ph.mark("collectives")
    idx, val = eng.serve_rank(table[:n * d].view(n, d), table[n * d:n * d + n], k, None)
    ph.mark("local_rank")
    gv, gi = eng._all_gather(val), eng._all_gather(idx)
    ph.mark("collectives")
    out = eng.serve_merge(gv, gi)
    ph.mark("merge")
    return out


def fold_rank_phased(eng, rows, items, rates, n, k, ph):
    """fold_in + rank_folded (rated items excluded) with the phases marked."""
    ph.mark("start")
    plan = eng.fold_plan(rows, items, rates, n)
    table = eng.fold_gather(plan["ids"])
    ph.mark("other")
    eng._all_reduce(table)
    ph.mark("collectives")
    folded = eng.fold_solve(plan, table)
    excl = eng.serve_exclusions(folded.ratings, torch.arange(n, dtype=torch.int32, device=eng.device))
    ph.mark("other")
    idx, val = eng.serve_rank(folded.feat, folded.bias, k, excl)
    ph.mark("local_rank")
    gv, gi = eng._all_gather(val), eng._all_gather(idx)
    ph.mark("collectives")
    out = eng.serve_merge(gv, gi)
    ph.mark("merge")
    return out


def timed_phases(fn, reps, warm=1):
    for _ in range(warm):
        fn(Phases())
    torch.cuda.synchronize()
    if dist.is_initialized():
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    tot, phs = {}, []
    e0.record()
    for _ in range(reps):
        ph = Phases()
        fn(ph)
        phs.append(ph)
    e1.record()
    torch.cuda.synchronize()
    for ph in phs:
        for k_, v in ph.split().items():
            tot[k_] = tot.get(k_, 0.0) + v / reps
    return dict(call_ms=e0.elapsed_time(e1) / reps, reps=reps, split_ms=tot)


def synthetic_ratings(n, I, seed):
    """n new users x N_RATINGS ratings, items skewed as bench_sharded draws them; the same on every rank."""
    rng = np.random.default_rng(seed)
    rows = np.repeat(np.arange(n, dtype=np.int32), N_RATINGS)
    u = rng.random(n * N_RATINGS)
    items = np.minimum((u * u * u * I).astype(np.int64), I - 1).astype(np.int32)
    rates = rng.integers(1, 6, n * N_RATINGS).astype(np.float32)
    return rows, items, rates


def same(a, b):
    return bool(torch.equal(a[0].cpu(), b[0].cpu()) and np.array_equal(a[1].cpu().numpy().view(np.int64),
                                                                        b[1].cpu().numpy().view(np.int64)))


def parity_multi(rank, world, dev):
    """Scaled-down configs[4] tables: the sharded calls against SvdEngine on rank 0's re-assembly, ids and bits."""
    U, I, d = bench_sharded.SHARDED["U"] // 1000, bench_sharded.SHARDED["I"] // 1000, bench_sharded.SHARDED["d"]
    eng = ShardedSvdEngine(U, I, d, LR, REG, rank, world, device=dev)
    rng = np.random.default_rng(5)
    users = rng.integers(0, U, 64).astype(np.int32)
    pu, pi = rng.integers(0, U, 200000).astype(np.int32), rng.integers(0, I, 200000).astype(np.int32)
    pu[:I], pi[:I] = users[0], np.arange(I)           # users[0]: every item excluded
    rows, items, rates = synthetic_ratings(64, I, 6)
    got_r = eng.rank_users(users, K, exclude=(pu, pi))
    folded = eng.fold_in(rows, items, rates)
    got_f = eng.rank_folded(folded, K)
    loc = eng.get_local_tables()
    parts = [None] * world
    dist.all_gather_object(parts, {k: loc[k] for k in ("user_feat", "item_feat", "user_bias", "item_bias", "mu")})
    res = None
    if rank == 0:
        tabs = {k: sharding.unshard_table([p[k] for p in parts]) for k in ("user_feat", "item_feat", "user_bias", "item_bias")}
        tabs["mu"] = parts[0]["mu"]
        ref = SvdEngine(U, I, d, LR, REG, tables=tabs, device=dev)
        want_f = ref.fold_in(rows, items, rates)
        fold_same = all(torch.equal(getattr(folded, x).view(torch.int32).cpu(), getattr(want_f, x).view(torch.int32).cpu())
                        for x in ("feat", "bias", "info"))
        res = dict(shape=dict(users=U, items=I, dim=d), world=world, queries=64, k=K, excluded_pairs=len(pu),
                   rank_users_identical=same(got_r, ref.rank_users(users, K, exclude=(pu, pi))),
                   fold_in_identical=fold_same, rank_folded_identical=same(got_f, ref.rank_folded(want_f, K)))
        res["pass"] = res["rank_users_identical"] and res["fold_in_identical"] and res["rank_folded_identical"]
        del ref
    dist.barrier()
    del eng
    torch.cuda.empty_cache()
    return res


def run_multi(args, rank, world, dev):
    out = dict(world=world)
    out["parity_scaled_down"] = parity_multi(rank, world, dev)
    w = bench_sharded.SHARDED
    eng = ShardedSvdEngine(w["U"], w["I"], w["d"], LR, REG, rank, world, device=dev)
    mine = dict(rank=rank, rank_users=[], fold_in_rank_folded=[])
    rng = np.random.default_rng(11)
    for n in (1, 64, 4096):
        q = eng._dev_i32(rng.integers(0, w["U"], n).astype(np.int32))
        r = timed_phases(lambda ph: rank_users_phased(eng, q, K, ph), args.reps if n < 4096 else max(args.reps // 4, 3))
        r["n"] = n
        mine["rank_users"].append(r)
    for n in (1, 4096):
        rows, items, rates = synthetic_ratings(n, w["I"], 12)
        r = timed_phases(lambda ph: fold_rank_phased(eng, rows, items, rates, n, K, ph),
                         args.reps if n < 4096 else max(args.reps // 4, 3))
        r["n"], r["ratings"] = n, n * N_RATINGS
        mine["fold_in_rank_folded"].append(r)
    parts = [None] * world
    dist.all_gather_object(parts, mine)
    out["config"] = bench_sharded.sharded_config(w, world)
    out["per_rank"] = parts
    return out


def run_world1(args, dev):
    from tf_recomm_b200 import init, synthetic
    U, I, _ = synthetic.SHAPES["ml25m"]
    d = 128
    tabs = init.init_tables(U, I, d, seed=3, bias_init="truncated_normal")
    ref = SvdEngine(U, I, d, LR, REG, tables=tabs, device=dev)
    eng = ShardedSvdEngine(U, I, d, LR, REG, 0, 1, tables=tabs, device=dev)
    out = dict(shape=dict(users=U, items=I, dim=d), k=K, queries=[])
    rng = np.random.default_rng(13)
    for n in (1, 64, 4096):
        q = eng._dev_i32(rng.integers(0, U, n).astype(np.int32))
        a, b = eng.rank_users(q, K), ref.rank_users(q, K)
        entry = dict(n=n, identical=same(a, b))
        reps = args.reps * (20 if n < 4096 else 2)
        sh, sv = [], []
        for _ in range(3):   # the public calls, alternated: sharded, single, sharded, ...
            sh.append(timed_phases(lambda ph: (ph.mark("start"), eng.rank_users(q, K), ph.mark("call")), reps)["call_ms"])
            sv.append(timed_phases(lambda ph: (ph.mark("start"), ref.rank_users(q, K), ph.mark("call")), reps)["call_ms"])
        entry["sharded_ms"] = sh
        entry["sharded_split_ms"] = timed_phases(lambda ph: rank_users_phased(eng, q, K, ph), reps)["split_ms"]
        entry["svd_engine_ms"] = sv
        entry["ratio_sharded_over_svd_engine"] = float(np.median(entry["sharded_ms"]) / np.median(sv))
        out["queries"].append(entry)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=12)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs CUDA devices; there is no CPU fallback"
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    name, power = gpu_info()
    res = dict(gpu=name, power_limit=power, n_gpus_visible=torch.cuda.device_count())
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
        res["multi"] = run_multi(args, rank, world, dev)
        dist.destroy_process_group()
    else:
        res["world1_ml25m"] = run_world1(args, dev)
    if rank == 0:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
        print(json.dumps(res))


if __name__ == "__main__":
    main()
