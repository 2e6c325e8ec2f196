"""Similar items and users: tfr_similar_rows (row_norms_kernel + similar_rows_score_kernel, then the select and merge of
csrc/rank_users.cu), SvdEngine.similar_items / similar_users, ShardedSvdEngine.similar_items / similar_users and
recommend.py --similar-items.

The oracle is numpy float64: the dot product and the squared norm summed over d in order from 0.0 (a loop over d of
vector adds; each product of two floats is exact in float64, as under the kernel's FMA), then np.sqrt and /, which are
correctly rounded as __dsqrt_rn and __ddiv_rn are.  Results must be equal bit for bit.

CPU: argument refusals and the workspace query, the registers of csrc/rank_users.cu, the instructions of
rank_users_score_kernel (pinned in tests/golden), and the sharded protocol over gloo at world 2, 3 and 4 with numpy
standing in for the kernels.  GPU: the kernel against the oracle at every tiling, chunk and pass edge, the engine
methods on every table layout and training path, G virtual ranks against SvdEngine, and the command line.
"""
import io
import os
import re
import subprocess

import numpy as np
import pytest
import torch

from tf_recomm_b200 import _lib, init, sharding

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NVCC = "/usr/local/cuda/bin/nvcc"
CUOBJDUMP = "/usr/local/cuda/bin/cuobjdump"
RANK_USERS = os.path.join(ROOT, "tf-recomm_b200", "csrc", "rank_users.cu")
LR, REG = 1e-3, 0.05
ADAM_FORK = _lib.FORK_FLAGS & ~_lib.OPT_SGD


# ---- numpy oracle ---------------------------------------------------------------------------------------------------------
def np_norms(X):
    s = np.zeros(X.shape[0])
    for j in range(X.shape[1]):
        x = X[:, j].astype(np.float64)
        s = s + x * x
    return np.sqrt(s)


def np_cosine(Q, V, abs_rows=False):
    """[n, N] float64 cosines of the rows of Q against the rows of V (NaN where a norm is zero)."""
    if abs_rows:
        Q, V = np.abs(Q), np.abs(V)
    with np.errstate(divide="ignore", invalid="ignore"):   # inf entries: 0 * inf and inf / inf are NaN, as on the device
        acc = np.zeros((Q.shape[0], V.shape[0]))
        for j in range(Q.shape[1]):
            acc = acc + Q[:, None, j].astype(np.float64) * V[None, :, j].astype(np.float64)
        den = np_norms(Q)[:, None] * np_norms(V)[None, :]
        s = acc / den
    s[den == 0] = np.nan
    return s


def np_rank_row(s, k, skip=-1):
    """Top k of one row of scores: finite scores only, not skip, score descending then id; padded with (-inf, -1)."""
    s = s.copy()
    if 0 <= skip < len(s):
        s[skip] = np.nan
    ids = np.nonzero(np.isfinite(s))[0]
    v = s[ids] + 0.0
    if len(ids) > k:   # keep every id at or above the k-th best score, then sort those
        t = np.partition(v, len(v) - k)[len(v) - k]
        keep = v >= t
        ids, v = ids[keep], v[keep]
    order = np.lexsort((ids, -v))[:k]
    out_v, out_i = np.full(k, -np.inf), np.full(k, -1, np.int32)
    out_v[:len(order)], out_i[:len(order)] = v[order], ids[order]
    return out_i, out_v


def np_similar(X, q, k, abs_rows=False):
    """The neighbours of rows q of X in X: (ids [n, k], scores [n, k])."""
    q = np.asarray(q)
    idx, val = np.full((len(q), k), -1, np.int32), np.full((len(q), k), -np.inf)
    step = max(1, min(64, (1 << 24) // X.shape[0]))   # queries per block: a few float64 [step, N] arrays at a time
    for a in range(0, len(q), step):
        sc = np_cosine(X[q[a:a + step]], X, abs_rows)
        for j in range(sc.shape[0]):
            idx[a + j], val[a + j] = np_rank_row(sc[j], k, int(q[a + j]))
    return idx, val


def assert_same(got, want, what=""):
    gi, gv = (x.cpu().numpy() if hasattr(x, "cpu") else x for x in got)
    wi, wv = want
    assert gi.shape == wi.shape, (what, gi.shape, wi.shape)
    bad = (gi != wi).any(axis=1)
    assert not bad.any(), "%s: %d rows differ, first %d" % (what, bad.sum(), np.nonzero(bad)[0][0])
    assert np.array_equal(gv.view(np.int64), wv.view(np.int64)), what


# ---- CPU ------------------------------------------------------------------------------------------------------------------
def test_workspace_query_needs_no_gpu():
    L = _lib.load()
    assert L.tfr_similar_rows_workspace_bytes(4096, 62423, 50) > L.tfr_rank_users_workspace_bytes(4096, 62423, 50)
    assert L.tfr_similar_rows_workspace_bytes(0, 62423, 50) > 0
    assert L.tfr_similar_rows_workspace_bytes(1, 0, 1) > 0
    for n, N, k in ((-1, 100, 10), (1, 100, 0), (1, 100, 1025), (1, -1, 10), (1, 1 << 31, 10)):
        assert L.tfr_similar_rows_workspace_bytes(n, N, k) < 0, (n, N, k)


def _call(L, dim=16, k=10, n=1, nq=100, N=200, qs=0, s=0, qf=1, q=1, f=1, val=1, idx=1, ws=1 << 30):
    """tfr_similar_rows with dummy (never dereferenced) pointers: only the argument checks can run."""
    p = 4096
    return L.tfr_similar_rows(qf and p, nq, qs, q and p, None, n, f and p, N, s, dim, 0, k, val and p, idx and p, p, ws,
                              None)


def test_invalid_arguments_are_refused_before_any_cuda_call():
    L = _lib.load()
    for kw in (dict(dim=0), dict(dim=513), dict(k=0), dict(k=1025), dict(n=-1), dict(n=1 << 31), dict(nq=-1),
               dict(nq=1 << 31), dict(N=-1), dict(N=1 << 31), dict(qs=15), dict(s=15), dict(qs=-1), dict(qf=0),
               dict(q=0), dict(f=0), dict(val=0), dict(idx=0)):
        assert _call(L, **kw) == -1, kw   # TFR_ERR_INVALID
    assert _call(L, ws=0) == -3           # TFR_ERR_WORKSPACE, before any launch
    assert _call(L, n=0, q=0, val=0, idx=0) == 0   # n_queries = 0: a no-op


def _compile(tmp_path):
    obj, log = str(tmp_path / "rank_users.o"), str(tmp_path / "ptxas.txt")
    with open(log, "w") as f:
        subprocess.check_call([NVCC, "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-ccbin",
                               "/usr/bin/g++", "-Xcompiler", "-fPIC", "-Xptxas", "-v", "-c", RANK_USERS, "-o", obj],
                              stdout=f, stderr=subprocess.STDOUT)
    return obj, log


@pytest.mark.skipif(not os.path.exists(NVCC), reason="needs the CUDA toolkit")
def test_similar_kernels_compile_without_stack_or_spills(tmp_path):
    from test_rank_users import _ptxas_lines
    _, log = _compile(tmp_path)
    info = _ptxas_lines(log)
    old = {"tfr::rank_users_score_kernel", "tfr::rank_users_select_kernel", "tfr::rank_users_merge_kernel"}
    new = {"void tfr::similar_rows_score_kernel<true>", "void tfr::similar_rows_score_kernel<false>",
           "tfr::row_norms_kernel"}
    assert old | new <= set(info), sorted(info)
    for name, (regs, stack, st, ld) in info.items():
        assert (stack, st, ld) == (0, 0, 0), (name, info[name])


def sass_listing(obj, mangled):
    """The instructions of one kernel from `cuobjdump -sass`, addresses and encodings dropped, one per line."""
    txt = subprocess.run([CUOBJDUMP, "-sass", obj], capture_output=True, text=True, check=True).stdout
    out, on = [], False
    for line in txt.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            on = m.group(1) == mangled
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(.*?)\s*;", line)
        if on and m:
            out.append(re.sub(r"\s+", " ", m.group(1)))
    return out


@pytest.mark.skipif(not os.path.exists(CUOBJDUMP), reason="needs the CUDA toolkit")
def test_rank_users_score_kernel_instructions_are_unchanged(tmp_path, golden_dir):
    """Sharing the scorer's main loop with similar_rows_score_kernel must not change rank_users_score_kernel: its
    instruction list is pinned as it was when the kernel had the loop to itself."""
    obj, _ = _compile(tmp_path)
    got = sass_listing(obj, "_ZN3tfr23rank_users_score_kernelEPKfS1_S1_S1_S1_iiillbPKiiPd")
    with open(os.path.join(golden_dir, "rank_users_score_kernel.sass")) as f:
        want = f.read().splitlines()
    assert len(got) > 100
    assert got == want


# ---- CPU: the sharded protocol over gloo ------------------------------------------------------------------------------------
def _protocol_tables(N, d):
    rng = np.random.default_rng(5)
    X = rng.standard_normal((N, d)).astype(np.float32)
    X[::4] = X[1]                    # duplicate rows across ranks: ties go by global id
    X[6] = 0.0                       # a zero row: queried and as a candidate
    X[9, ::2] = -0.0
    return X, np.r_[1, 6, 9, 2, 2, N - 1, 0, 5]


def _protocol_rank(rank, world, port, N, d, k, q):
    import torch.distributed as dist
    from test_sharded_serving import np_merge
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    X, ids = _protocol_tables(N, d)
    loc = sharding.shard_table(X, world, rank)
    N_loc = sharding.rows_on_rank(N, world, rank)
    n = len(ids)
    # 1. owner-filled query rows, all-reduced
    keys = sharding.local_keys(ids, world, rank, N_loc)
    mine = keys < N_loc
    g = np.zeros((n, d), np.float32)
    g[mine] = loc[keys[mine]]
    t = torch.from_numpy(g.ravel().copy())
    dist.all_reduce(t)
    g = t.numpy().reshape(n, d)
    # 2. cosine against the local shard, the query's own row skipped where this rank owns it
    sc = np_cosine(g, loc)
    val, idx = np.empty((n, k)), np.empty((n, k), np.int32)
    for j, i in enumerate(ids):
        idx[j], val[j] = np_rank_row(sc[j], k, i // world if i % world == rank else -1)
    # 3. all-gather, merge
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
def test_sharded_similar_protocol_equals_full_table(world):
    import torch.multiprocessing as mp
    from test_sharded_serving import _free_port
    N, d, k = 31, 7, 12
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_protocol_rank, args=(r, world, port, N, d, k, q)) for r in range(world)]
    for p in procs:
        p.start()
    got_v, got_i = q.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    X, ids = _protocol_tables(N, d)
    want_i, want_v = np_similar(X, ids, k)
    assert np.array_equal(got_i, want_i), world
    assert np.array_equal(got_v.view(np.int64), want_v.view(np.int64)), world
    assert np.all(got_i[1] == -1)               # the zero row ranks nothing
    assert not (got_i == 6).any()               # and is nobody's neighbour
    for j, i in enumerate(ids):
        assert i not in got_i[j]


# ---- GPU: the kernel against the oracle ---------------------------------------------------------------------------------------
def _tables(U, I, d, seed=21):
    tabs = init.init_tables(U, I, d, seed=seed, bias_init="truncated_normal")
    tabs["user_feat"] *= 25
    tabs["item_feat"] *= 25
    return tabs


def _engine(U, I, d, flags=0, tabs=None, seed=21):
    from tf_recomm_b200.engine import SvdEngine
    tabs = _tables(U, I, d, seed) if tabs is None else tabs
    return SvdEngine(U, I, d, LR, REG, flags=flags, tables=tabs), tabs


def _special(X):
    """Zero rows, -0.0 entries, an exact duplicate and a row with an inf, in place."""
    X[3] = 0.0
    X[5, ::3] = -0.0
    X[8] = X[2]
    X[11] = -0.0
    X[13, 1 % X.shape[1]] = np.inf
    return X


def _queries(N, rng, n=40):
    q = np.r_[rng.integers(0, N, n - 8), 2, 8, 3, 5, 11, 13, 0, N - 1].astype(np.int32)
    return q[rng.permutation(len(q))]


@pytest.fixture
def rank_chunk():
    old = _lib.tune_get("RANK_CHUNK")
    yield lambda v: _lib.tune_set("RANK_CHUNK", v)
    _lib.tune_set("RANK_CHUNK", old)


@pytest.mark.gpu
@pytest.mark.parametrize("d", [1, 3, 31, 32, 33, 127, 128, 129, 512])
def test_similar_items_and_users_match_numpy(d):
    """Items (I = 1100, so k = 1024 is a real k) and users (U = 260); k = 1, 50, rows - 1, rows and 1024 (clamped);
    zero rows, -0.0, duplicates, an inf entry; repeated and unordered ids."""
    U, I = 260, 1100
    rng = np.random.default_rng(d)
    tabs = _tables(U, I, d)
    _special(tabs["item_feat"])
    _special(tabs["user_feat"])
    eng, _ = _engine(U, I, d, tabs=tabs)
    for name, X, fn in (("items", tabs["item_feat"], eng.similar_items), ("users", tabs["user_feat"], eng.similar_users)):
        N = X.shape[0]
        q = _queries(N, rng)
        for k in (k for k in (1, 50, N - 1, N, 1024) if min(k, N) <= 1024):   # k of the table is at most 1024
            kk = min(k, N)
            want = np_similar(X, q, kk)
            got = fn(q, k=k)
            assert_same(got, want, "%s d=%d k=%d" % (name, d, k))
            gi = got[0].cpu().numpy()
            assert not (gi == q[:, None]).any()          # never the query itself
            assert (gi[q == 3] == -1).all() and (gi[q == 11] == -1).all()   # zero rows rank nothing
            assert not np.isin(gi, [3, 11, 13]).any()    # and zero / non-finite rows are nobody's neighbour
            assert (gi[q == 13] == -1).all()


@pytest.mark.gpu
@pytest.mark.parametrize("chunk", [1024, 4096])
def test_chunk_and_tile_edges(rank_chunk, chunk):
    """Candidate rows at the 128-row tile and selection-chunk edges, query counts at the 32-row block edges."""
    rank_chunk(chunk)
    d = 5
    rng = np.random.default_rng(chunk)
    for N in sorted({127, 128, 129, 257, chunk - 1, chunk, chunk + 1, 2 * chunk + 1}):
        X = _special(rng.standard_normal((N, d)).astype(np.float32))
        eng, _ = _engine(64, N, d, tabs=dict(_tables(64, N, d), item_feat=X))
        for n in (1, 31, 32, 33):
            q = rng.integers(0, N, n).astype(np.int32)
            for k in (1, 50, min(N, 1024)):
                assert_same(eng.similar_items(q, k), np_similar(X, q, min(k, N)), "N=%d n=%d k=%d" % (N, n, k))


@pytest.mark.gpu
def test_two_scoring_passes():
    """2^21 + 3 candidates: a pass holds 64 queries' scores, so 70 queries take two passes."""
    N, d, k = (1 << 21) + 3, 2, 50
    rng = np.random.default_rng(3)
    X = rng.standard_normal((N, d)).astype(np.float32)
    X[::7] = X[5]
    eng, _ = _engine(64, N, d, tabs=dict(_tables(64, 64, d), item_feat=X, item_bias=np.zeros(N, np.float32)))
    q = np.r_[rng.integers(0, N, 66), 5, 5, 12, N - 1].astype(np.int32)
    assert_same(eng.similar_items(q, k), np_similar(X, q, k), "two passes")


@pytest.mark.gpu
def test_out_of_range_ids():
    from tf_recomm_b200.engine import TfrError
    U, I, d, k = 50, 300, 16, 10
    eng, tabs = _engine(U, I, d)
    for bad in ([3, I], [-1], torch.tensor([2, I + 5], device=eng.device)):
        with pytest.raises(TfrError):
            eng.similar_items(bad, k)
    with pytest.raises(TfrError):
        eng.similar_users([U], k)
    assert eng.similar_items([], k)[0].shape == (0, k)
    assert eng.similar_items(torch.tensor([4, 9], device=eng.device), 400)[0].shape == (2, I)
    # C level: ids out of range in the middle of the list give (-inf, -1) rows and are never read through
    q = torch.tensor([4, 9, I, 17, -3, 1 << 30, 4], dtype=torch.int32, device=eng.device)
    idx, val = eng._similar_rows(eng.t["item_feat"], I, eng.feat_stride, q, q, eng.t["item_feat"], I, False, k)
    idx, val = idx.cpu().numpy(), val.cpu().numpy()
    qn = q.cpu().numpy()
    ok = (qn >= 0) & (qn < I)
    assert (idx[~ok] == -1).all() and np.isneginf(val[~ok]).all()
    assert_same((idx[ok], val[ok]), np_similar(tabs["item_feat"], qn[ok], k))


def _train_batches(rng, U, I, n, binary=False):
    users, items = rng.integers(0, U, n).astype(np.int32), rng.integers(0, I, n).astype(np.int32)
    rates = (rng.integers(0, 2, n) if binary else rng.integers(1, 6, n)).astype(np.float32)
    return users, items, rates


@pytest.mark.gpu
@pytest.mark.parametrize("flags", [0, _lib.OPT_SGD, _lib.ABS_ITEM, ADAM_FORK, _lib.FORK_FLAGS])
def test_layouts_and_fork_model_after_steps(flags):
    """Adam (stride 3d) and SGD (stride d) layouts, the fork model (|q_i| on the item side), before and after steps."""
    U, I, d, k = 300, 700, 24, 30
    rng = np.random.default_rng(flags)
    eng, _ = _engine(U, I, d, flags=flags)
    abs_items = bool(flags & _lib.ABS_ITEM)
    for step in range(2):
        if step:
            for _ in range(4):
                eng.train_step(*_train_batches(rng, U, I, 2000, binary=bool(flags & _lib.LOSS_SIGMOID_CE)))
        T = eng.get_tables()
        qi, qu = _queries(I, rng), _queries(U, rng)
        assert_same(eng.similar_items(qi, k), np_similar(T["item_feat"], qi, k, abs_items), "items flags=%d" % flags)
        assert_same(eng.similar_users(qu, k), np_similar(T["user_feat"], qu, k), "users flags=%d" % flags)


@pytest.mark.gpu
def test_after_als_and_ials_sweeps():
    U, I, d, k = 200, 500, 16, 20
    rng = np.random.default_rng(9)
    users, items, rates = _train_batches(rng, U, I, 5000)
    eng, _ = _engine(U, I, d)
    eng.als_sweep(eng.als_data(users, items, rates))
    T = eng.get_tables()
    qi, qu = _queries(I, rng), _queries(U, rng)
    assert_same(eng.similar_items(qi, k), np_similar(T["item_feat"], qi, k), "ALS items")
    assert_same(eng.similar_users(qu, k), np_similar(T["user_feat"], qu, k), "ALS users")
    eng, _ = _engine(U, I, d)
    eng.ials_sweep(eng.ials_data(users, items), 10.0)
    T = eng.get_tables()
    assert_same(eng.similar_items(qi, k), np_similar(T["item_feat"], qi, k), "iALS items")
    assert_same(eng.similar_users(qu, k), np_similar(T["user_feat"], qu, k), "iALS users")


# ---- GPU: G virtual ranks -----------------------------------------------------------------------------------------------------
def similar_virtual(engs, ids, k, items):
    from test_sharded_serving import _all_reduce, _merge
    e0 = engs[0]
    q = e0._dev_i32(np.asarray(ids))
    k = min(k, e0.I if items else e0.U)
    tables = _all_reduce([e.similar_gather(q, items) for e in engs])
    return _merge(engs, [e.similar_rank(t, q, k, items) for e, t in zip(engs, tables)])


@pytest.mark.gpu
@pytest.mark.parametrize("G", [1, 2, 3, 4, 5, 8])
@pytest.mark.parametrize("flags", [0, _lib.ABS_ITEM])
def test_sharded_similar_bit_identical_to_one_gpu(G, flags):
    """Both tables, signed zeros (the all-reduce turns an owned -0.0 into +0.0), zero rows, duplicates across ranks."""
    from test_sharded_serving import _engines
    U, I, d = 61, 203, 33
    rng = np.random.default_rng(G + flags)
    tabs = _tables(U, I, d)
    _special(tabs["item_feat"])
    _special(tabs["user_feat"])
    tabs["item_feat"][::5] = tabs["item_feat"][1]
    engs, ref = _engines(G, U, I, d, tabs, flags)
    for items, N, fn in ((True, I, ref.similar_items), (False, U, ref.similar_users)):
        q = _queries(N, rng)
        for k in (1, 50, N - 1, N):
            assert_same(similar_virtual(engs, q, k, items), tuple(x.cpu().numpy() for x in fn(q, k)),
                        "G=%d items=%s k=%d" % (G, items, k))


@pytest.mark.gpu
def test_sharded_world_one_public_methods():
    import torch.distributed as dist
    from test_sharded_serving import _engines
    assert not dist.is_initialized()
    U, I, d = 80, 150, 15
    rng = np.random.default_rng(1)
    (eng,), ref = _engines(1, U, I, d, _tables(U, I, d))
    for k in (1, 10, I + 1):
        qi, qu = _queries(I, rng), _queries(U, rng)
        assert_same(eng.similar_items(qi, k), tuple(x.cpu().numpy() for x in ref.similar_items(qi, k)), "k=%d" % k)
        assert_same(eng.similar_users(qu, k), tuple(x.cpu().numpy() for x in ref.similar_users(qu, k)), "k=%d" % k)
    assert eng.similar_items([], 5)[0].shape == (0, 5)
    with pytest.raises(_lib.TfrError, match="out of range"):
        eng.similar_items([I])


# ---- recommend.py ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_recommend_similar_items(tmp_path):
    import recommend
    from tf_recomm_b200.engine import SvdEngine
    eng, _ = _engine(70, 400, 12)
    ckpt = str(tmp_path / "model.ckpt")
    eng.save(ckpt)
    items = [3, 17, 42, 3, 399]
    buf = io.StringIO()
    recommend.main(["--checkpoint", ckpt, "--similar-items", ",".join(map(str, items)), "--k", "7"], out=buf)
    idx, val = SvdEngine.from_checkpoint(ckpt).similar_items(items, k=7)
    idx, val = idx.cpu().numpy(), val.cpu().numpy()
    want = "".join("%d\t%s\n" % (i, " ".join("%d:%.6f" % (j, v) for j, v in zip(ri, rv) if j >= 0))
                   for i, ri, rv in zip(items, idx, val))
    assert buf.getvalue() == want
