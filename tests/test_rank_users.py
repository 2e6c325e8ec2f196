"""Exact float64 top-k for a batch of query users: tfr_rank_users (score / select / merge kernels of csrc/rank_users.cu),
SvdEngine.rank_users and SvdEngine.from_checkpoint above it, and the recommend.py command line."""
import ctypes as C
import io
import os
import re
import subprocess
import sys
from contextlib import redirect_stdout

import numpy as np
import pytest

from tf_recomm_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NVCC = "/usr/local/cuda/bin/nvcc"


# ---- numpy reference (as in test_rank_unseen.py) ---------------------------------------------------------------------------
def ref_rank_excluding(M, k, excluded):
    """The float64 ranking of M (score descending, lowest id on ties) with each row's excluded items removed; ranks past
    the row's rankable items are (-inf, -1)."""
    U, I = M.shape
    idx = np.full((U, k), -1, np.int32)
    val = np.full((U, k), -np.inf)
    for u in range(U):
        keep = np.ones(I, bool)
        keep[list(excluded[u])] = False
        cand = np.nonzero(keep)[0]
        order = cand[np.lexsort((cand, -M[u, cand]))][:k]
        idx[u, :len(order)] = order
        val[u, :len(order)] = M[u, order]
    return idx, val


# ---- CPU -------------------------------------------------------------------------------------------------------------------
def test_workspace_query_needs_no_gpu():
    L = _lib.load()
    assert L.tfr_rank_users_workspace_bytes(4096, 62423, 50) > 0
    assert L.tfr_rank_users_workspace_bytes(0, 62423, 50) > 0
    assert L.tfr_rank_users_workspace_bytes(1, 0, 1) > 0
    assert L.tfr_rank_users_workspace_bytes(1, 100, 1024) > 0
    for n, I, k in ((-1, 100, 10), (1, 100, 0), (1, 100, 1025), (1, -1, 10)):
        assert L.tfr_rank_users_workspace_bytes(n, I, k) < 0, (n, I, k)


def _call(L, dim=16, k=10, n=1, val=1, idx=1, q=1):
    """tfr_rank_users with dummy (never dereferenced) pointers: only the argument checks can run."""
    p = 4096
    return L.tfr_rank_users(p, p, p, p, p, 100, 200, dim, 0, 0, 0, q and p, n, k, None, None, val and p, idx and p, p,
                            1 << 30, None)


def test_invalid_arguments_are_refused_before_any_cuda_call():
    L = _lib.load()
    for kw in (dict(dim=0), dict(dim=513), dict(k=0), dict(k=1025), dict(val=0), dict(idx=0), dict(q=0)):
        assert _call(L, **kw) == -1, kw   # TFR_ERR_INVALID
    assert _call(L, n=0, val=0, idx=0, q=0) == 0   # n_queries = 0: a no-op


def _ptxas_lines(path):
    """{kernel (demangled, parameters dropped): (registers, stack, spill stores, spill loads)} from `-Xptxas -v`."""
    out, cur = {}, None
    for line in open(path):
        m = re.search(r"Function properties for (\S+)", line)
        if m:
            cur = subprocess.run(["c++filt", m.group(1)], capture_output=True, text=True).stdout.strip().split("(")[0]
        m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and cur:
            out.setdefault(cur, [None, *(int(x) for x in m.groups())])
        m = re.search(r"Used (\d+) registers", line)
        if m and cur:
            out[cur][0] = int(m.group(1))
    return out


@pytest.mark.skipif(not os.path.exists(NVCC), reason="needs the CUDA toolkit")
def test_rank_users_kernels_compile_without_spills(tmp_path):
    obj, log = str(tmp_path / "rank_users.o"), str(tmp_path / "ptxas.txt")
    with open(log, "w") as f:
        subprocess.check_call([NVCC, "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-ccbin",
                               "/usr/bin/g++", "-Xcompiler", "-fPIC", "-Xptxas", "-v", "-c",
                               os.path.join(ROOT, "tf-recomm_b200", "csrc", "rank_users.cu"), "-o", obj],
                              stdout=f, stderr=subprocess.STDOUT)
    info = _ptxas_lines(log)
    names = {"tfr::rank_users_score_kernel", "tfr::rank_users_select_kernel", "tfr::rank_users_merge_kernel"}
    assert names <= set(info), sorted(info)
    for name, (regs, stack, st, ld) in info.items():
        assert (stack, st, ld) == (0, 0, 0), (name, info[name])


# ---- GPU -------------------------------------------------------------------------------------------------------------------
def _engine(U, I, d, ties=0, seed=21, flags=0):
    from tf_recomm_b200 import init
    from tf_recomm_b200.engine import SvdEngine
    tabs = init.init_tables(U, I, d, seed=seed, bias_init="truncated_normal")
    tabs["user_feat"] *= 25; tabs["item_feat"] *= 25
    if ties:
        tabs["item_bias"][::ties] = tabs["item_bias"][0]
        tabs["item_feat"][::ties] = tabs["item_feat"][0]
    return SvdEngine(U, I, d, 1e-3, 0.05, flags=flags, tables=tabs), tabs


def _f64_scores(tabs):
    U64, V64 = tabs["user_feat"].astype(np.float64), tabs["item_feat"].astype(np.float64)
    return ((U64 @ V64.T + tabs["user_bias"].astype(np.float64)[:, None]) + tabs["item_bias"].astype(np.float64)[None, :]) \
        + float(tabs["mu"][0])


def _exclusion_pairs(U, I, kk, seed=0):
    """Random pairs with duplicates; user 0: every item; user 1: I - kk + 3 items (fewer than kk rankable); the last three
    users: nothing.  -> (users, items) shuffled, and the per-user sets."""
    rng = np.random.default_rng(seed)
    n1 = min(I - kk + 3, I - 1)
    users, items = rng.integers(0, U, 4 * U), rng.integers(0, I, 4 * U)
    users, items = np.concatenate([users, users[:50]]), np.concatenate([items, items[:50]])
    keep = (users > 1) & (users < U - 3)
    x1 = rng.choice(I, n1, replace=False)
    users = np.concatenate([users[keep], np.zeros(I, np.int64), np.ones(n1 + len(x1[:5]), np.int64)]).astype(np.int32)
    items = np.concatenate([items[keep], np.arange(I), x1, x1[:5]]).astype(np.int32)
    perm = rng.permutation(len(users))
    users, items = users[perm], items[perm]
    sets = [set() for _ in range(U)]
    for u, i in zip(users, items):
        sets[u].add(int(i))
    return users, items, sets


def _queries(U, seed=1):
    """Shuffled, with duplicates, and users 0 and 1 (all excluded / fewer than k rankable) in it."""
    rng = np.random.default_rng(seed)
    q = np.concatenate([rng.integers(0, U, 40), [0, 1, 1, U - 1, 0]]).astype(np.int32)
    return q[rng.permutation(len(q))]


@pytest.fixture
def rank_chunk():
    """Sets the RANK_CHUNK knob for a test and restores it afterwards."""
    old = _lib.tune_get("RANK_CHUNK")
    yield lambda v: _lib.tune_set("RANK_CHUNK", v)
    _lib.tune_set("RANK_CHUNK", old)


def _same(a, b):
    """(items, float64 scores) pairs equal in ids and in bit patterns."""
    ai, av = (x.cpu().numpy() if hasattr(x, "cpu") else x for x in a)
    bi, bv = (x.cpu().numpy() if hasattr(x, "cpu") else x for x in b)
    assert ai.shape == bi.shape, (ai.shape, bi.shape)
    bad = (ai != bi).any(axis=1)
    assert not bad.any(), "%d rows differ, first %d" % (bad.sum(), np.nonzero(bad)[0][0])
    assert np.array_equal(av.view(np.int64), bv.view(np.int64))


@pytest.mark.gpu
@pytest.mark.parametrize("U,I,d,k,ties", [(300, 2500, 64, 50, 0), (129, 3000, 128, 10, 5), (150, 2200, 15, 50, 0),
                                          (100, 1500, 20, 1, 3), (120, 1800, 160, 10, 0), (257, 40, 32, 50, 0),
                                          (90, 2100, 128, 50, 1)])
@pytest.mark.parametrize("masked", [False, True])
def test_rank_users_is_bit_identical_to_rank_all_users(rank_chunk, U, I, d, k, ties, masked):
    """rank_users(q)[j] = rank_all_users()[q[j]] in item ids and float64 bits: tcgen05 dims (64, 128; 32 with I < k) and
    exact-path dims (15, 20, 160), tied items, k = 1 / 10 / 50, a user with every item excluded, one with fewer than k
    rankable items; the chunk size 1024 and the default."""
    eng, _ = _engine(U, I, d, ties)
    kk = min(k, I)
    excl = None
    if masked:
        users, items, _ = _exclusion_pairs(U, I, kk)
        excl = eng.pair_csr(users, items)
        ref = eng.rank_all_users(k=k, exclude=excl)
    elif d % 32 == 0 and d <= 128:
        ref = eng.rank_all_users(k=k)
    else:
        ref = eng._rank_excluding(k, None, None)   # nothing excluded, any dim
    q = _queries(U)
    want = (ref[0].cpu().numpy()[q], ref[1].cpu().numpy()[q])
    if masked:
        assert (want[0][q == 0] == -1).all() and ((want[0][q == 1] == -1).any() or kk <= 3)
    for chunk in (1024, 4096):
        rank_chunk(chunk)
        _same(eng.rank_users(q, k=k, exclude=excl), want)


@pytest.mark.gpu
@pytest.mark.parametrize("masked", [False, True])
def test_rank_users_matches_numpy_float64_ranking(masked):
    U, I, d, k = 80, 1300, 48, 20
    eng, tabs = _engine(U, I, d, ties=7)
    M = _f64_scores(tabs)
    sets = [set() for _ in range(U)]
    excl = None
    if masked:
        users, items, sets = _exclusion_pairs(U, I, k)
        excl = (users, items)
    q = _queries(U)
    idx, val = eng.rank_users(q, k=k, exclude=excl)
    ref_idx, ref_val = ref_rank_excluding(M, k, sets)
    assert np.array_equal(idx.cpu().numpy(), ref_idx[q])
    np.testing.assert_allclose(val.cpu().numpy(), ref_val[q], rtol=1e-12, atol=1e-12)


@pytest.mark.gpu
@pytest.mark.parametrize("d", [64, 20])
def test_rank_users_of_the_fork_model(d):
    """ABS_ITEM: ranked by u.|v| + biases, the same bits as rank_all_users on the same fork engine."""
    U, I, k = 200, 1600, 20
    eng, _ = _engine(U, I, d, flags=_lib.FORK_FLAGS)
    users, items, _ = _exclusion_pairs(U, I, k)
    excl = eng.pair_csr(users, items)
    q = _queries(U)
    ref = eng.rank_all_users(k=k, exclude=excl)
    _same(eng.rank_users(q, k=k, exclude=excl), (ref[0].cpu().numpy()[q], ref[1].cpu().numpy()[q]))


@pytest.mark.gpu
def test_chunk_size_does_not_change_results(rank_chunk):
    U, I, d, k = 64, 9000, 128, 50
    eng, _ = _engine(U, I, d, ties=4)
    users, items, _ = _exclusion_pairs(U, I, k)
    excl = eng.pair_csr(users, items)
    q = _queries(U)
    outs = []
    for chunk in (1024, 3072, 16384):
        rank_chunk(chunk)
        outs.append(tuple(x.cpu().numpy() for x in eng.rank_users(q, k=k, exclude=excl)))
    for o in outs[1:]:
        _same(outs[0], o)


def _c_rank(eng, q_dev, k, excl=None, ws=None, stream=None):
    """tfr_rank_users straight from the C ABI on device query ids -> (idx, val, workspace)."""
    import torch
    n = q_dev.numel()
    idx = torch.empty(n, k, dtype=torch.int32, device=eng.device)
    val = torch.empty(n, k, dtype=torch.float64, device=eng.device)
    nbytes = eng.L.tfr_rank_users_workspace_bytes(n, eng.I, k)
    if ws is None:
        ws = torch.empty(nbytes, dtype=torch.uint8, device=eng.device)
    T = eng.t
    st = stream if stream is not None else torch.cuda.current_stream(eng.device).cuda_stream
    _lib.check(eng.L.tfr_rank_users(T["user_feat"].data_ptr(), T["item_feat"].data_ptr(), T["user_bias"].data_ptr(),
                                    T["item_bias"].data_ptr(), T["mu"].data_ptr(), eng.U, eng.I, eng.d, eng.feat_stride,
                                    eng.feat_stride, eng.flags, q_dev.data_ptr(), n, k,
                                    excl.indptr.data_ptr() if excl is not None else None,
                                    excl.items.data_ptr() if excl is not None else None, val.data_ptr(), idx.data_ptr(),
                                    ws.data_ptr(), nbytes, st))
    return idx, val, ws


@pytest.mark.gpu
def test_edge_cases():
    import torch
    from tf_recomm_b200.engine import TfrError
    U, I, d, k = 50, 1200, 32, 10
    eng, _ = _engine(U, I, d)
    ref = eng.rank_all_users(k=k)
    _same(eng.rank_users(7, k=k), (ref[0].cpu().numpy()[[7]], ref[1].cpu().numpy()[[7]]))        # n = 1
    idx, val = eng.rank_users(np.zeros(0, np.int32), k=k)                                          # n = 0
    assert tuple(idx.shape) == (0, k) and tuple(val.shape) == (0, k)
    for bad in ([3, U], [-1], torch.tensor([2, U + 5], device=eng.device)):
        with pytest.raises(TfrError):
            eng.rank_users(bad, k=k)
    # C level: ids out of range in the middle of the list give (-inf, -1) rows; the other rows are unchanged
    q = np.array([4, 9, U, 17, -3, 1 << 30, 4], np.int32)
    idx, val, _ = _c_rank(eng, torch.from_numpy(q).to(eng.device), k)
    idx, val = idx.cpu().numpy(), val.cpu().numpy()
    ok = (q >= 0) & (q < U)
    assert (idx[~ok] == -1).all() and np.isneginf(val[~ok]).all()
    _same((idx[ok], val[ok]), (ref[0].cpu().numpy()[q[ok]], ref[1].cpu().numpy()[q[ok]]))


@pytest.mark.gpu
def test_graph_capture_and_replay_with_new_query_ids():
    import torch
    U, I, d, k = 120, 2500, 64, 20
    eng, _ = _engine(U, I, d)
    users, items, _ = _exclusion_pairs(U, I, k)
    excl = eng.pair_csr(users, items)
    rng = np.random.default_rng(5)
    q_dev = torch.from_numpy(rng.integers(0, U, 33).astype(np.int32)).to(eng.device)
    cap = torch.cuda.Stream(device=eng.device)
    cap.wait_stream(torch.cuda.current_stream(eng.device))
    exe = C.c_void_p()
    with torch.cuda.stream(cap):
        _lib.check(eng.L.tfr_graph_begin_capture(cap.cuda_stream))
        try:
            g_idx, g_val, _ = _c_rank(eng, q_dev, k, excl, stream=cap.cuda_stream)
        finally:
            rc = eng.L.tfr_graph_end_capture(cap.cuda_stream, C.byref(exe))
        _lib.check(rc)
    torch.cuda.current_stream(eng.device).wait_stream(cap)
    try:
        new = rng.integers(0, U, 33).astype(np.int32)
        q_dev.copy_(torch.from_numpy(new))
        _lib.check(eng.L.tfr_graph_launch(exe, torch.cuda.current_stream(eng.device).cuda_stream))
        torch.cuda.synchronize(eng.device)
        _same((g_idx, g_val), eng.rank_users(new, k=k, exclude=excl))
    finally:
        eng.L.tfr_graph_destroy(exe)


@pytest.mark.gpu
@pytest.mark.parametrize("d", [128, 15])
def test_every_user_at_the_ml1m_shape(d):
    """The synthetic ML-1M shape (6040 x 3952), every user a query, the training split excluded: the same bits as
    rank_all_users(exclude=train)."""
    from tf_recomm_b200 import config, synthetic
    from tf_recomm_b200.engine import SvdEngine
    U, I, N = synthetic.SHAPES["ml1m"]
    users, items, rates = synthetic.make_ratings(U, I, N, seed=config.SEED)
    (tu, ti, _), _ = synthetic.split(users, items, rates)
    eng = SvdEngine(U, I, d, 1e-3, 0.05, device_init_seed=7)
    excl = eng.pair_csr(tu, ti)
    ref = eng.rank_all_users(k=50, exclude=excl)
    _same(eng.rank_users(np.arange(U), k=50, exclude=excl), ref[:2])


# ---- recommend.py ------------------------------------------------------------------------------------------------------------
def _parse(text):
    out = []
    for line in text.splitlines():
        u, _, rest = line.partition("\t")
        pairs = [p.split(":") for p in rest.split()]
        out.append((int(u), [int(i) for i, _ in pairs], [float(v) for _, v in pairs]))
    return out


@pytest.mark.gpu
def test_recommend_cli(tmp_path):
    import svd_train_val
    import recommend
    from tf_recomm_b200 import config, synthetic
    from tf_recomm_b200.engine import SvdEngine
    ckpt = str(tmp_path / "model.ckpt")
    data = ["--synthetic", "ml1m", "--ratings", "20000"]
    with redirect_stdout(io.StringIO()):
        svd_train_val.main(data + ["--epochs", "1", "--dim", "20", "--checkpoint", ckpt, "--logdir", str(tmp_path / "log")])
    users = [3, 17, 42, 3, 6039]
    run = subprocess.run([sys.executable, os.path.join(ROOT, "recommend.py"), "--checkpoint", ckpt, "--users",
                          ",".join(map(str, users)), "--k", "10"] + data, capture_output=True, text=True, cwd=ROOT)
    assert run.returncode == 0, run.stderr
    lines = _parse(run.stdout)
    assert [u for u, _, _ in lines] == users
    U, I, _ = synthetic.SHAPES["ml1m"]
    au, ai, ar = synthetic.make_ratings(U, I, 20000, seed=config.SEED)
    (tu, ti, _), _ = synthetic.split(au, ai, ar)
    eng = SvdEngine.from_checkpoint(ckpt)
    assert (eng.U, eng.I, eng.d) == (U, I, 20)
    for excluded, text in ((True, run.stdout), (False, None)):
        if text is None:
            buf = io.StringIO()
            recommend.main(["--checkpoint", ckpt, "--users", ",".join(map(str, users)), "--k", "10", "--no-exclude"] + data,
                           out=buf)
            text = buf.getvalue()
        idx, val = eng.rank_users(users, k=10, exclude=(tu, ti) if excluded else None)
        idx, val = idx.cpu().numpy(), val.cpu().numpy()
        for r, (u, items, scores) in enumerate(_parse(text)):
            keep = idx[r] >= 0
            assert items == idx[r][keep].tolist()
            np.testing.assert_allclose(scores, val[r][keep], rtol=0, atol=5.1e-7)
            seen = set(ti[tu == u].tolist())
            if excluded:
                assert not seen & set(items)
