"""Serving from row-sharded tables (ShardedSvdEngine.rank_users / fold_in / rank_folded): exact top-k and fold-in with the
item table spread over G ranks, ids and bits equal to SvdEngine on the re-assembled tables.

CPU: the merge of the per-rank lists (tfr_shard_topk_merge) mirrored in numpy and checked against a brute-force sort of
the union on hand-built lists; the whole protocol (gather + all-reduce + per-rank ranking + all-gather + merge) over gloo
at world 2, 3 and 4 with numpy float64 standing in for the kernels; the argument refusals of the new ABI entries; and the
registers of csrc/shard_rank.cu.

GPU: G virtual ranks on one GPU, the collectives emulated as test_sharded_geometry does (all-reduce = a sum of the
buffers, all-gather = a stack), tables injected through tables=.  Every rank must return the same bits, and those must
be SvdEngine's.
"""
import os
import socket
import subprocess

import numpy as np
import pytest
import torch

from tf_recomm_b200 import _lib, init, sharding

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NVCC = "/usr/local/cuda/bin/nvcc"
SHARD_RANK = os.path.join(ROOT, "tf-recomm_b200", "csrc", "shard_rank.cu")
LR, REG = 1e-3, 0.05
ADAM_FORK = _lib.FORK_FLAGS & ~_lib.OPT_SGD    # sharded tables train with Adam only


# ---- the merge, in numpy ----------------------------------------------------------------------------------------------------
def np_merge(val, idx):
    """tfr_shard_topk_merge in numpy: val / idx [G, n, k] sorted per-rank lists of local ids (-1 ends a list) -> the top k
    of the union under (score descending, global id ascending), global id = local * G + g, padded with (-inf, -1)."""
    G, n, k = idx.shape
    out_v, out_i = np.full((n, k), -np.inf), np.full((n, k), -1, np.int32)
    for q in range(n):
        h = [0] * G
        for r in range(k):
            best = None
            for g in range(G):
                if h[g] < k and idx[g, q, h[g]] >= 0:
                    cand = (val[g, q, h[g]], int(idx[g, q, h[g]]) * G + g, g)
                    if best is None or cand[0] > best[0] or (cand[0] == best[0] and cand[1] < best[1]):
                        best = cand
            if best is None:
                break
            out_v[q, r], out_i[q, r] = best[0], best[1]
            h[best[2]] += 1
    return out_v, out_i


def np_rank(scores, k, excluded=()):
    """The exact ranking of one row of float64 scores: score descending, id ascending, excluded ids left out; k columns
    padded with (-inf, -1).  -0.0 and +0.0 are one score and come back as +0.0, as in tfr_rank_users."""
    ids = np.array([i for i in range(len(scores)) if i not in set(excluded)], np.int64)
    v = scores[ids] + 0.0
    order = np.lexsort((ids, -v))[:k]
    out_v, out_i = np.full(k, -np.inf), np.full(k, -1, np.int32)
    out_v[:len(order)], out_i[:len(order)] = v[order], ids[order]
    return out_v, out_i


def merge_cases():
    """(name, val [G, n, k], idx [G, n, k]) hand-built lists: ties across ranks, exhausted and all -1 lists, G = 1 and 8."""
    cases = []
    rng = np.random.default_rng(7)
    for G, n, k in ((1, 3, 4), (2, 4, 5), (3, 5, 7), (8, 6, 9), (8, 2, 1), (5, 3, 40)):
        val = np.full((G, n, k), -np.inf)
        idx = np.full((G, n, k), -1, np.int32)
        for g in range(G):
            for q in range(n):
                m = int(rng.integers(0, k + 1)) if q else k   # query 0: full lists; others: exhausted after m
                if q == n - 1 and g % 2:
                    m = 0                                      # all -1 lists
                loc = np.sort(rng.choice(50, m, replace=False))
                v = rng.choice([2.5, 1.0, 0.0, -1.0, -3.75], m)   # few values: ties inside and across ranks
                order = np.lexsort((loc, -v))
                val[g, q, :m], idx[g, q, :m] = v[order], loc[order]
        cases.append(("G%d_n%d_k%d" % (G, n, k), val, idx))
    val = np.full((4, 1, 3), 7.0)                               # every score equal: global id order alone
    idx = np.array([[[0, 1, 2]], [[0, 1, 2]], [[0, 1, 2]], [[0, 1, 2]]], np.int32)
    cases.append(("all_tied", val, idx))
    cases.append(("all_empty", np.full((3, 2, 4), -np.inf), np.full((3, 2, 4), -1, np.int32)))
    return cases


# ---- CPU ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,val,idx", merge_cases(), ids=[c[0] for c in merge_cases()])
def test_merge_reference_is_the_top_k_of_the_union(name, val, idx):
    G, n, k = idx.shape
    got_v, got_i = np_merge(val, idx)
    for q in range(n):
        ent = [(val[g, q, j], int(idx[g, q, j]) * G + g) for g in range(G) for j in range(k) if idx[g, q, j] >= 0]
        ent.sort(key=lambda e: (-e[0], e[1]))
        ent = ent[:k]
        want_v = np.array([e[0] for e in ent] + [-np.inf] * (k - len(ent)))
        want_i = np.array([e[1] for e in ent] + [-1] * (k - len(ent)), np.int32)
        assert np.array_equal(got_i[q], want_i), (name, q)
        assert np.array_equal(got_v[q], want_v), (name, q)


def test_new_abi_entries_refuse_bad_arguments():
    """Every refusal comes before any CUDA call (dummy pointers are never read; no GPU here)."""
    L = _lib.load()
    p = 256

    def merge(G=2, n=4, k=3, val=p, idx=p, ov=p, oi=p):
        return L.tfr_shard_topk_merge(val, idx, G, n, k, ov, oi, None)
    for kw in (dict(G=0), dict(G=9), dict(k=0), dict(k=1025), dict(n=-1), dict(n=1 << 31), dict(val=None), dict(idx=None),
               dict(ov=None), dict(oi=None)):
        assert merge(**kw) == -1, kw
    assert merge(n=0, val=None, idx=None, ov=None, oi=None) == 0   # n = 0: a no-op

    def excl(fn, G=2, rank=0, n=4, n_rows=10, indptr=p, rows=p, out=p):
        if fn == "indptr":
            return L.tfr_shard_excl_indptr(indptr, p, n_rows, rows, n, G, rank, out, p, 1 << 20, None)
        return L.tfr_shard_excl_fill(indptr, p, n_rows, rows, n, G, rank, out, p, None)
    for fn in ("indptr", "fill"):
        for kw in (dict(G=0), dict(G=9), dict(rank=-1), dict(rank=2), dict(n=-1), dict(n=1 << 31), dict(n_rows=-1),
                   dict(n_rows=1 << 31), dict(indptr=None), dict(rows=None), dict(out=None)):
            assert excl(fn, **kw) == -1, (fn, kw)
    assert excl("fill", n=0, indptr=None, rows=None) == 0
    assert L.tfr_shard_excl_workspace_bytes(-1) == -1
    assert L.tfr_shard_excl_indptr(p, p, 10, p, 4, 2, 0, p, p, 0, None) == -3   # TFR_ERR_WORKSPACE, before any launch


@pytest.mark.skipif(not os.path.exists(NVCC), reason="needs the CUDA toolkit")
def test_shard_rank_kernels_compile_without_stack_or_spills(tmp_path):
    from test_rank_users import _ptxas_lines
    obj, log = str(tmp_path / "shard_rank.o"), str(tmp_path / "ptxas.txt")
    with open(log, "w") as f:
        subprocess.check_call([NVCC, "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-ccbin",
                               "/usr/bin/g++", "-Xcompiler", "-fPIC", "-Xptxas", "-v", "-c", SHARD_RANK, "-o", obj],
                              stdout=f, stderr=subprocess.STDOUT)
    info = _ptxas_lines(log)
    names = {"tfr::shard_topk_merge_kernel", "tfr::shard_excl_count_kernel", "tfr::shard_excl_fill_kernel"}
    assert names <= set(info), sorted(info)
    for name, (regs, stack, st, ld) in info.items():
        assert (stack, st, ld) == (0, 0, 0), (name, info[name])


# ---- CPU: the protocol over gloo -----------------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _f64_scores(uf, ub, vf, ib, mu):
    """((acc + b_u) + b_i) + mu with acc summed over d in order from 0.0, as tfr_rank_users scores."""
    acc = np.zeros((uf.shape[0], vf.shape[0]))
    for j in range(uf.shape[1]):
        acc = acc + uf[:, None, j].astype(np.float64) * vf[None, :, j].astype(np.float64)
    return ((acc + ub.astype(np.float64)[:, None]) + ib.astype(np.float64)[None, :]) + np.float64(mu)


def _protocol_tables(U, I, d):
    tabs = init.init_tables(U, I, d, seed=3, bias_init="truncated_normal")
    tabs["item_feat"][::3] = tabs["item_feat"][0]     # ties across ranks
    tabs["item_bias"][::3] = tabs["item_bias"][0]
    rng = np.random.default_rng(4)
    pu, pi = rng.integers(0, U, 200), rng.integers(0, I, 200)
    pu, pi = np.r_[pu, np.full(I, 5)], np.r_[pi, np.arange(I)]   # user 5: every item excluded
    return tabs, np.r_[5, 2, 2, 0, 9, 1, 5, 3], pu, pi


def _protocol_rank(rank, world, port, U, I, d, k, q):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    tabs, users, pu, pi = _protocol_tables(U, I, d)
    loc = {n: sharding.shard_table(tabs[n], world, rank) for n in ("user_feat", "user_bias", "item_feat", "item_bias")}
    U_loc = sharding.rows_on_rank(U, world, rank)
    n = len(users)
    # 1. owner-filled query rows; 2. all-reduce
    keys = sharding.local_keys(users, world, rank, U_loc)
    mine = keys < U_loc
    g_uf, g_ub = np.zeros((n, d), np.float32), np.zeros(n, np.float32)
    g_uf[mine], g_ub[mine] = loc["user_feat"][keys[mine]], loc["user_bias"][keys[mine]]
    flat = torch.from_numpy(np.concatenate([g_uf.ravel(), g_ub]))
    dist.all_reduce(flat)
    flat = flat.numpy()
    g_uf, g_ub = flat[:n * d].reshape(n, d), flat[n * d:]
    # 3. per-rank ranking of the local items, exclusions as local ids
    sc = _f64_scores(g_uf, g_ub, loc["item_feat"], loc["item_bias"], tabs["mu"][0])
    val, idx = np.empty((n, k)), np.empty((n, k), np.int32)
    for j, u in enumerate(users):
        ex = [i // world for i in pi[pu == u] if i % world == rank]
        val[j], idx[j] = np_rank(sc[j], k, ex)
    # 4. all-gather; 5. merge
    outs = []
    for a in (val, idx):
        parts = [torch.empty_like(torch.from_numpy(a)) for _ in range(world)]
        dist.all_gather(parts, torch.from_numpy(a))
        outs.append(torch.stack(parts).numpy())
    got_v, got_i = np_merge(*outs)
    if rank == 0:
        q.put((got_v, got_i))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3, 4])
def test_sharded_ranking_protocol_equals_full_table_ranking(world):
    import torch.multiprocessing as mp
    U, I, d, k = 13, 29, 6, 12
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_protocol_rank, args=(r, world, port, U, I, d, k, q)) for r in range(world)]
    for p in procs:
        p.start()
    got_v, got_i = q.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    tabs, users, pu, pi = _protocol_tables(U, I, d)
    sc = _f64_scores(tabs["user_feat"][users], tabs["user_bias"][users], tabs["item_feat"], tabs["item_bias"], tabs["mu"][0])
    for j, u in enumerate(users):
        want_v, want_i = np_rank(sc[j], k, pi[pu == u])
        assert np.array_equal(got_i[j], want_i), (world, j)
        assert np.array_equal(got_v[j].view(np.int64), want_v.view(np.int64)), (world, j)
    assert np.all(got_i[0] == -1)   # user 5: every item excluded


# ---- GPU: G virtual ranks ------------------------------------------------------------------------------------------------------
def _tables(U, I, d, seed=21, ties=3):
    tabs = init.init_tables(U, I, d, seed=seed, bias_init="truncated_normal")
    tabs["user_feat"] *= 25
    tabs["item_feat"] *= 25
    if ties:
        tabs["item_bias"][::ties] = tabs["item_bias"][0]
        tabs["item_feat"][::ties] = tabs["item_feat"][0]
    return tabs


def _engines(G, U, I, d, tabs, flags=0):
    from tf_recomm_b200.engine import SvdEngine
    from tf_recomm_b200.sharded import ShardedSvdEngine
    engs = [ShardedSvdEngine(U, I, d, LR, REG, rank=r, world=G, tables=tabs, flags=flags) for r in range(G)]
    return engs, SvdEngine(U, I, d, LR, REG, flags=flags, tables=tabs)


def _all_reduce(bufs):
    """What NCCL's sum computes on the owner-filled buffers (one non-zero term per element); nothing at world 1."""
    if len(bufs) == 1:
        return bufs
    total = torch.stack(bufs).sum(0)
    return [total.clone() for _ in bufs]


def _merge(engs, lists):
    """lists[r] = rank r's (local idx, val); every rank merges the all-gathered lists and must get the same bits."""
    gi = torch.stack([x[0] for x in lists])
    gv = torch.stack([x[1] for x in lists])
    outs = [e.serve_merge(gv.clone(), gi.clone()) for e in engs]
    for r, (i, v) in enumerate(outs[1:], 1):
        assert torch.equal(i, outs[0][0]) and torch.equal(v.view(torch.int64), outs[0][1].view(torch.int64)), "rank %d" % r
    return outs[0]


def rank_virtual(engs, users, k, exclude=None):
    """ShardedSvdEngine.rank_users on len(engs) virtual ranks; exclude: global (users, items) pairs."""
    e0 = engs[0]
    q = e0._dev_i32(np.asarray(users))
    n, d, k = q.numel(), e0.d, min(k, e0.I)
    tables = _all_reduce([e.serve_gather(q) for e in engs])
    lists = []
    for e, t in zip(engs, tables):
        excl = e.serve_exclusions(e.pair_csr(*exclude), q) if exclude is not None else None
        lists.append(e.serve_rank(t[:n * d].view(n, d), t[n * d:n * d + n], k, excl))
    return _merge(engs, lists)


def fold_virtual(engs, rows, items, rates, n=None, reg=None):
    plans = [e.fold_plan(rows, items, rates, n, reg) for e in engs]
    tables = _all_reduce([e.fold_gather(p["ids"]) for e, p in zip(engs, plans)])
    outs = [e.fold_solve(p, t) for e, p, t in zip(engs, plans, tables)]
    for r, o in enumerate(outs[1:], 1):
        for a, b in zip((o.feat, o.bias, o.info), (outs[0].feat, outs[0].bias, outs[0].info)):
            assert torch.equal(a.view(torch.int32), b.view(torch.int32)), "rank %d" % r
    return outs[0]


def rank_folded_virtual(engs, folded, k, exclude_rated=True):
    n = folded.feat.shape[0]
    rows = torch.arange(n, dtype=torch.int32, device=engs[0].device)
    k = min(k, engs[0].I)
    lists = [e.serve_rank(folded.feat, folded.bias, k, e.serve_exclusions(folded.ratings, rows) if exclude_rated else None)
             for e in engs]
    return _merge(engs, lists)


def assert_same_ranking(got, want, what):
    gi, gv = (x.cpu().numpy() for x in got)
    wi, wv = (x.cpu().numpy() for x in want)
    assert gi.shape == wi.shape, (what, gi.shape, wi.shape)
    assert np.array_equal(gi, wi), what
    assert np.array_equal(gv.view(np.int64), wv.view(np.int64)), what


def _pairs(rng, U, I, full_user, dense_user):
    """Training pairs with duplicates, one user with every item and one with all but 3."""
    pu, pi = rng.integers(0, U, 6 * U), rng.integers(0, I, 6 * U)
    pu = np.r_[pu, pu[:50], np.full(I, full_user), np.full(I - 3, dense_user)]
    pi = np.r_[pi, pi[:50], np.arange(I), rng.permutation(I)[:I - 3]]
    return pu.astype(np.int32), pi.astype(np.int32)


def _queries(rng, U, full_user, dense_user):
    return np.r_[rng.integers(0, U, 30), 7, 7, full_user, dense_user, 0, U - 1, 3].astype(np.int32)


GRID_G = [1, 2, 3, 4, 5, 8]
GRID_D = [1, 3, 4, 32, 33, 128, 129, 256, 512]


@pytest.mark.gpu
@pytest.mark.parametrize("d", GRID_D)
@pytest.mark.parametrize("G", GRID_G)
def test_rank_users_bit_identical_to_one_gpu(G, d):
    """I = 203 (k up to I and past it) and I = 1031 (k = 1024); neither divisible by any G > 1.  Query ids repeat and come
    in any order; no exclusion, and the training pairs (with duplicates) excluded, among them a user with every item and
    one with fewer rankable items than k."""
    U = 61
    for I in (203, 1031):
        rng = np.random.default_rng(G * 1000 + d + I)
        tabs = _tables(U, I, d)
        engs, ref = _engines(G, U, I, d, tabs)
        pu, pi = _pairs(rng, U, I, 11, 12)
        users = _queries(rng, U, 11, 12)
        I_loc = sharding.rows_on_rank(I, G, 0)
        ks = {1, 50, I_loc - 1, I_loc, I_loc + 1} | ({I, I + 5} if I < 1024 else {1024})
        csr_ref = ref.pair_csr(pu, pi)
        for k in sorted(x for x in ks if 1 <= min(x, I) <= 1024):
            what = "G=%d d=%d I=%d k=%d" % (G, d, I, k)
            assert_same_ranking(rank_virtual(engs, users, k), ref.rank_users(users, k), what)
            got = rank_virtual(engs, users, k, exclude=(pu, pi))
            assert_same_ranking(got, ref.rank_users(users, k, exclude=csr_ref), what + " excluded")
            assert np.all(got[0].cpu().numpy()[users == 11] == -1), what


@pytest.mark.gpu
@pytest.mark.parametrize("G", [2, 3, 5])
def test_rank_users_fork_model_and_trained_tables(G):
    """ABS_ITEM (u.|v| + biases), and tables taken after sharded train_step_a2a steps (the interleaved Adam layout, a
    trained mu) re-assembled for the single-GPU reference."""
    from test_gpu_parity import _a2a_emulated_step, make_batch
    from test_sharded_geometry import _tables as assembled
    from tf_recomm_b200.engine import SvdEngine
    U, I, d = 97, 301, 33
    rng = np.random.default_rng(G)
    pu, pi = _pairs(rng, U, I, 4, 9)
    users = _queries(rng, U, 4, 9)
    for flags in (_lib.ABS_ITEM, ADAM_FORK, 0):
        tabs = _tables(U, I, d)
        engs, ref = _engines(G, U, I, d, tabs, flags)
        if flags != _lib.ABS_ITEM:   # train a few steps; the reference takes the re-assembled tables
            for _ in range(3):
                _a2a_emulated_step(engs, *make_batch(rng, U, I, 700, binary=bool(flags & _lib.LOSS_SIGMOID_CE)))
            got_tabs = assembled(engs)
            assert got_tabs["mu"][0] != tabs["mu"][0]
            ref = SvdEngine(U, I, d, LR, REG, flags=flags, tables=got_tabs)
        for k in (1, 50, 120):
            what = "G=%d flags=%d k=%d" % (G, flags, k)
            assert_same_ranking(rank_virtual(engs, users, k), ref.rank_users(users, k), what)
            assert_same_ranking(rank_virtual(engs, users, k, exclude=(pu, pi)), ref.rank_users(users, k, exclude=(pu, pi)),
                                what + " excluded")


def _signed_zero_tables(U, I, d):
    tabs = _tables(U, I, d, ties=0)
    tabs["user_feat"][::5, ::2] = -0.0
    tabs["user_feat"][3] = -0.0
    tabs["item_feat"][::4, 1::3] = -0.0
    tabs["item_feat"][7] = -0.0
    tabs["user_bias"][::3] = -0.0
    tabs["item_bias"][::2] = -0.0
    assert np.signbit(tabs["user_bias"][0]) and np.signbit(tabs["item_feat"][7, 0])
    return tabs


@pytest.mark.gpu
@pytest.mark.parametrize("G", [1, 2, 3])
def test_signed_zeros_give_the_same_bits(G):
    """The all-reduce turns an owned -0.0 into +0.0 (G > 1; at G = 1 nothing is reduced and -0.0 stays): the results
    must not change, since every float64 sum of the scorer and of the Gram starts from +0.0."""
    U, I, d = 40, 57, 9
    tabs = _signed_zero_tables(U, I, d)
    engs, ref = _engines(G, U, I, d, tabs)
    users = np.r_[3, 0, 1, 2, 3, 15, 39].astype(np.int32)
    for k in (1, 20, 57):
        assert_same_ranking(rank_virtual(engs, users, k), ref.rank_users(users, k), "G=%d k=%d" % (G, k))
    rows = np.r_[0, 0, 1, 1, 1, 2, 3, 3].astype(np.int32)
    items = np.r_[7, 4, 7, 8, 0, 7, 12, 16].astype(np.int32)       # item 7 all -0.0, items 4 / 8 / 12 / 16 partly
    rates = np.r_[3, 4, 5, 1, 2, 4, 5, 3].astype(np.float32)
    got, want = fold_virtual(engs, rows, items, rates), ref.fold_in(rows, items, rates)
    for a, b in zip((got.feat, got.bias, got.info), (want.feat, want.bias, want.info)):
        assert torch.equal(a.view(torch.int32), b.view(torch.int32)), G
    assert_same_ranking(rank_folded_virtual(engs, got, 10), ref.rank_folded(want, 10), "folded G=%d" % G)


def _assert_same_folded(got, want, what):
    for name in ("feat", "bias", "info"):
        a, b = getattr(got, name), getattr(want, name)
        assert a.shape == b.shape, (what, name)
        assert torch.equal(a.view(torch.int32), b.view(torch.int32)), (what, name)
    assert torch.equal(got.ratings.indptr, want.ratings.indptr) and torch.equal(got.ratings.items, want.ratings.items), what


@pytest.mark.gpu
@pytest.mark.parametrize("d", [1, 4, 33, 128])
@pytest.mark.parametrize("G", [1, 2, 3, 8])
@pytest.mark.parametrize("flags", [0, _lib.REG_BIAS, _lib.ABS_ITEM | _lib.REG_BIAS])
def test_fold_in_and_rank_folded_bit_identical_to_one_gpu(flags, G, d):
    """Rows without ratings (row 2 and the rows past the last label), a row whose items all live on rank 0, duplicate
    ratings; rank_folded with and without the rated items excluded."""
    U, I = 50, 211
    rng = np.random.default_rng(G * 100 + d + flags)
    tabs = _tables(U, I, d)
    engs, ref = _engines(G, U, I, d, tabs, flags)
    rows = np.r_[rng.integers(0, 2, 60), np.full(9, 3), rng.integers(4, 9, 80), 0, 0].astype(np.int32)
    items = np.r_[rng.integers(0, I, 60), G * np.arange(9), rng.integers(0, I, 80), 5, 5].astype(np.int32)
    rates = rng.integers(1, 6, len(rows)).astype(np.float32)
    for n in (None, 12):
        what = "flags=%d G=%d d=%d n=%s" % (flags, G, d, n)
        got, want = fold_virtual(engs, rows, items, rates, n=n), ref.fold_in(rows, items, rates, n=n)
        _assert_same_folded(got, want, what)
        assert int(want.info.abs().sum()) == 0
        for k in (1, 50, I):
            for ex in (True, False):
                assert_same_ranking(rank_folded_virtual(engs, got, k, ex), ref.rank_folded(want, k, ex),
                                    "%s k=%d exclude_rated=%s" % (what, k, ex))


@pytest.mark.gpu
def test_fold_in_refusals():
    from tf_recomm_b200.sharded import ShardedSvdEngine
    U, I, d = 30, 40, 8
    tabs = _tables(U, I, d)
    eng = ShardedSvdEngine(U, I, d, LR, REG, rank=1, world=3, tables=tabs, flags=ADAM_FORK)
    with pytest.raises(_lib.TfrError, match="sigmoid cross-entropy"):
        eng.fold_in([0], [1], [3.0])
    eng = ShardedSvdEngine(U, I, d, LR, REG, rank=1, world=3, tables=tabs)
    with pytest.raises(_lib.TfrError, match="reg must be >= 0"):
        eng.fold_in([0], [1], [3.0], reg=-1.0)
    with pytest.raises(_lib.TfrError, match="differ in length"):
        eng.fold_in([0, 1], [1], [3.0])
    with pytest.raises(_lib.TfrError, match="out of range"):
        eng.fold_in([0], [I], [3.0])
    with pytest.raises(_lib.TfrError, match="out of range"):
        eng.fold_in([0, 4], [1, 2], [3.0, 1.0], n=3)
    with pytest.raises(_lib.TfrError, match="out of range"):
        eng.rank_users([0, U])
    with pytest.raises(_lib.TfrError, match="out of range"):
        eng.rank_users([0], exclude=([0], [I]))


@pytest.mark.gpu
@pytest.mark.parametrize("d", [15, 128])
def test_world_one_public_methods_match_svd_engine(d):
    """At world 1 with no process group the public methods run without torch.distributed."""
    import torch.distributed as dist
    assert not dist.is_initialized()
    U, I = 80, 150
    rng = np.random.default_rng(d)
    tabs = _tables(U, I, d)
    (eng,), ref = _engines(1, U, I, d, tabs)
    pu, pi = _pairs(rng, U, I, 2, 3)
    users = _queries(rng, U, 2, 3)
    for k in (1, 50, I + 1):
        assert_same_ranking(eng.rank_users(users, k), ref.rank_users(users, k), "k=%d" % k)
        assert_same_ranking(eng.rank_users(users, k, exclude=(pu, pi)), ref.rank_users(users, k, exclude=(pu, pi)),
                            "k=%d excluded" % k)
        assert_same_ranking(eng.rank_users(users, k, exclude=eng.pair_csr(pu, pi)),
                            ref.rank_users(users, k, exclude=(pu, pi)), "k=%d pair_csr" % k)
    assert eng.rank_users([], 5)[0].shape == (0, 5)
    rows, items = rng.integers(0, 6, 90).astype(np.int32), rng.integers(0, I, 90).astype(np.int32)
    rates = rng.integers(1, 6, 90).astype(np.float32)
    got, want = eng.fold_in(rows, items, rates), ref.fold_in(rows, items, rates)
    _assert_same_folded(got, want, "world 1")
    for ex in (True, False):
        assert_same_ranking(eng.rank_folded(got, 40, ex), ref.rank_folded(want, 40, ex), "folded %s" % ex)


@pytest.mark.gpu
@pytest.mark.parametrize("name,val,idx", merge_cases(), ids=[c[0] for c in merge_cases()])
def test_merge_kernel_matches_reference(name, val, idx):
    L = _lib.load()
    G, n, k = idx.shape
    v, i = torch.from_numpy(val).cuda(), torch.from_numpy(idx).cuda()
    ov, oi = torch.empty(n, k, dtype=torch.float64, device="cuda"), torch.empty(n, k, dtype=torch.int32, device="cuda")
    _lib.check(L.tfr_shard_topk_merge(v.data_ptr(), i.data_ptr(), G, n, k, ov.data_ptr(), oi.data_ptr(),
                                      torch.cuda.current_stream().cuda_stream))
    want_v, want_i = np_merge(val, idx)
    assert np.array_equal(oi.cpu().numpy(), want_i), name
    assert np.array_equal(ov.cpu().numpy().view(np.int64), want_v.view(np.int64)), name


@pytest.mark.gpu
@pytest.mark.parametrize("G", [1, 3, 8])
def test_exclusion_lists_match_reference(G):
    """tfr_shard_excl_indptr / _fill: query rows (repeated, out of range, empty) of a CSR with duplicates, every rank."""
    from tf_recomm_b200.engine import PairCSR
    from tf_recomm_b200.sharded import ShardedSvdEngine
    rng = np.random.default_rng(G)
    n_rows, I = 20, 300
    lens = rng.integers(0, 70, n_rows)
    lens[4] = 0
    indptr = np.r_[0, np.cumsum(lens)].astype(np.int64)
    items = np.concatenate([np.sort(rng.integers(0, I, m)) for m in lens]).astype(np.int32)
    rows = np.r_[3, 3, 4, 19, 0, 7, 25, -1, 11].astype(np.int32)
    csr = PairCSR(torch.from_numpy(indptr).cuda(), torch.from_numpy(items).cuda())
    for r in range(G):
        eng = ShardedSvdEngine(40, I, 4, LR, REG, rank=r, world=G)
        got = eng.serve_exclusions(csr, torch.from_numpy(rows).cuda())
        want = [items[indptr[x]:indptr[x + 1]] if 0 <= x < n_rows else np.zeros(0, np.int32) for x in rows]
        want = [w[w % G == r] // G for w in want]
        assert np.array_equal(got.indptr.cpu().numpy(), np.r_[0, np.cumsum([len(w) for w in want])]), (G, r)
        assert np.array_equal(got.items.cpu().numpy(), np.concatenate(want)), (G, r)
