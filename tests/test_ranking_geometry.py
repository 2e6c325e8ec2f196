"""The exact float64 rankings at every geometry they can reach, bit for bit against an in-order reference: tfr_rank_users
(csrc/rank_users.cu: score, select and merge kernels, the path of rank_users, rank_folded and recommend.py), the exact
paths of rank_all_users (allpairs_exact_rows_kernel, allpairs_rescore_kernel) and tfr_topk_rows (get_ranking).

The header defines a score exactly: ((acc + b_u) + b_i) + mu in float64, acc summed over d = 0 .. dim-1 in that order
from 0.0 of (double)u[d] * (double)v[d].  Each product of two fp32 values is exact in float64 and numpy rounds every add
to nearest, so inorder_scores below is that definition, and it equals the kernels' FMA chain bit for bit.  A BLAS matmul
sums in an order of its own (OpenBLAS splits the dims into panels past a few hundred), so a reference built on one can
only be trusted to a tolerance; this one is compared in bits.

tfr_rank_users splits the item axis into chunks of RANK_CHUNK items (rounded to a multiple of RU_MIN_CHUNK, clamped to
[RU_MIN_CHUNK, RU_MAX_CHUNK]), takes the exact top-k of every (query, chunk) by a radix select whose ties at the
threshold are taken RU_SEL_THREADS positions at a time, sorts the survivors bitonically (padded to a power of two up to
RU_MAX_K), and merges the chunk lists with one warp per query, lane l holding lists l, l + 32, ...  Queries are scored in
passes of at most RU_SCORE_BUDGET bytes of float64.  The GPU sweeps reach every k class up to 1024, every dim class up to
512, more than one pass, more than 32 lists per merge lane and a last chunk shorter than k; the CPU tests mirror the
chunk and pass arithmetic against tfr_rank_users_workspace_bytes and check that the sweeps reach those classes.
"""
import math
import os
import re

import numpy as np
import pytest

from tf_recomm_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "tf-recomm_b200", "csrc")


def _source(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


def _constant(src, name):
    m = re.search(r"constexpr int [^;]*\b%s = (\d+)" % name, _source(src))
    assert m, (src, name)
    return int(m.group(1))


RU_QB = _constant("rank_users.cu", "RU_QB")
RU_SEL_THREADS = _constant("rank_users.cu", "RU_SEL_THREADS")
RU_MIN_CHUNK = _constant("rank_users.cu", "RU_MIN_CHUNK")
RU_MAX_CHUNK = _constant("rank_users.cu", "RU_MAX_CHUNK")
RU_MAX_K = _constant("rank_users.cu", "RU_MAX_K")
RU_SCORE_BUDGET = 1 << int(re.search(r"RU_SCORE_BUDGET = \(int64_t\)1 << (\d+);", _source("rank_users.cu")).group(1))
RANK_CHUNK_DEFAULT = int(re.search(r'\{"RANK_CHUNK", (-?\d+)\}', _source("capi.cu")).group(1))
AP_MAX_CAND = _constant("allpairs.cu", "AP_MAX_CAND")

# ---- the sweeps (the GPU tests run exactly these; the CPU mirror checks what they reach) -------------------------------
CHUNKS = (1024, RANK_CHUNK_DEFAULT)
DIMS = [1, 2, 31, 32, 33, 63, 64, 65, 127, 128, 129, 255, 256, 257, 383, 511, 512]
FORK_DIMS = [1, 33, 128, 257, 512]            # ABS_ITEM (u.|v|) on the fork's SGD layout
DIM_QUERIES, DIM_K = 40, 100


def dim_items(d):
    """1500 .. 2999 items, a different tail past the last chunk and item tile at every dim"""
    return 1500 + (d * 389) % 1500


KS = [1, 2, 31, 32, 33, 128, 129, 255, 256, 257, 511, 512, 513, 1023, 1024]
K_ITEMS, K_QUERIES, K_DIM = 3000, 40, 40      # 3000 = 2 * 1024 + 952: at chunk 1024 the last chunk is short of k >= 953
ITEM_COUNTS = [1023, 1024, 1025, 4095, 4096, 4097, 16384, 16385]
ITEM_KS = (33, 1024)
FEW_ITEMS = [1, 5, 100, 1000]                 # called with k = n_items + 1 and k = 1024
TIE_CASES = [("all", 5000), ("straddle", 3000), ("flat_chunk", 3000)]
TIE_KS = (1, 257, 1024)
KNOBS = [1024, 3000, 16384, 100000, 0, -7]
KNOB_ITEMS, KNOB_K = 40000, 300
MERGE_ITEMS, MERGE_KS = [40961, 69000], (50, 1024)
MP_QUERIES, MP_ITEMS, MP_DIM, MP_K = 300, 1 << 20, 4, 64


def ru_chunk_items(knob):
    """rank_users.cu ru_chunk_items"""
    c = min(max(knob, RU_MIN_CHUNK), RU_MAX_CHUNK)
    return (c + RU_MIN_CHUNK - 1) // RU_MIN_CHUNK * RU_MIN_CHUNK


def ru_pass_queries(n, n_items):
    """rank_users.cu ru_pass_queries: queries scored per pass"""
    nb = max(RU_SCORE_BUDGET // (n_items * 8 if n_items > 0 else 8), 1)
    return min(nb, 65535 * RU_QB, n)


def ru_workspace(n, n_items, k):
    """tfr_rank_users_workspace_bytes"""
    a = lambda x: (x + 255) // 256 * 256
    parts = n * ((n_items + RU_MIN_CHUNK - 1) // RU_MIN_CHUNK) * k
    return 256 + a(ru_pass_queries(n, n_items) * n_items * 8) + a(parts * 8) + a(parts * 4) + \
        a(n * ((n_items + RU_MIN_CHUNK - 1) // RU_MIN_CHUNK) * 4)


def sweep_calls():
    """(n_queries, n_items, k, RANK_CHUNK knob) of every tfr_rank_users call of the GPU tests below (k as passed to the C
    ABI: the engine clamps it to n_items)."""
    calls = []
    for d in DIMS + FORK_DIMS:
        calls += [(DIM_QUERIES, dim_items(d), DIM_K, c) for c in CHUNKS]
    calls += [(K_QUERIES, K_ITEMS, k, c) for k in KS for c in CHUNKS]
    calls += [(_item_queries(n), n, k, c) for n in ITEM_COUNTS for k in ITEM_KS for c in CHUNKS]
    calls += [(20, n, k, c) for n in FEW_ITEMS for k in (n + 1, RU_MAX_K) for c in CHUNKS]
    calls += [(24, n, k, c) for _, n in TIE_CASES for k in TIE_KS for c in CHUNKS]
    calls += [(16, KNOB_ITEMS, KNOB_K, c) for c in KNOBS]
    calls += [(8, n, k, 1024) for n in MERGE_ITEMS for k in MERGE_KS]
    calls += [(MP_QUERIES, MP_ITEMS, MP_K, c) for c in CHUNKS]
    calls += [(min(128, MP_QUERIES - s), MP_ITEMS, MP_K, RANK_CHUNK_DEFAULT) for s in range(0, MP_QUERIES, 128)]
    return calls


def _item_queries(n_items):
    return 40 if n_items < 10000 else 24


# ---- reference -----------------------------------------------------------------------------------------------------------
def inorder_scores(U, V, bu, bi, mu, abs_item=False):
    """float64 scores [len(U), len(V)] as the header defines them: acc = 0.0, acc = acc + u[d] * v[d] for d = 0 .. dim-1
    (each product exact), then ((acc + b_u) + b_i) + mu; abs_item: v = |v|."""
    U64 = np.asarray(U, np.float32).astype(np.float64)
    V64 = np.asarray(V, np.float32).astype(np.float64)
    if abs_item:
        V64 = np.abs(V64)
    acc = np.zeros((U64.shape[0], V64.shape[0]))
    for d in range(U64.shape[1]):
        acc = acc + U64[:, d, None] * V64[None, :, d]
    bu64 = np.asarray(bu, np.float32).astype(np.float64)
    bi64 = np.asarray(bi, np.float32).astype(np.float64)
    return ((acc + bu64[:, None]) + bi64[None, :]) + float(np.float32(mu))


def ref_rank(S, k, excluded=None):
    """Every row of S ranked (score descending, lowest id on ties), excluded[r] (ids, duplicates allowed) and NaN removed,
    padded with (-inf, -1) -> (ids int32 [n, k], values [n, k] of S's dtype)."""
    n, I = S.shape
    idx = np.full((n, k), -1, np.int32)
    val = np.full((n, k), -np.inf, S.dtype)
    for r in range(n):
        keep = ~np.isnan(S[r])
        if excluded is not None:
            keep[np.asarray(excluded[r], np.int64)] = False
        cand = np.nonzero(keep)[0]
        order = cand[np.lexsort((cand, -S[r, cand]))][:k]
        idx[r, :len(order)], val[r, :len(order)] = order, S[r, order]
    return idx, val


def assert_same(got, want, what=""):
    """ids equal and values equal in bit patterns"""
    gi, gv = (x.cpu().numpy() if hasattr(x, "cpu") else np.asarray(x) for x in got)
    wi, wv = want
    assert gi.shape == wi.shape, (what, gi.shape, wi.shape)
    bad = np.argwhere((gi != wi) | (gv.view(np.int64 if gv.itemsize == 8 else np.int32) !=
                                    wv.view(np.int64 if wv.itemsize == 8 else np.int32)))
    if len(bad):
        r, c = bad[0]
        raise AssertionError("%s: %d entries differ, first row %d rank %d: got (%d, %r), want (%d, %r)" %
                             (what, len(bad), r, c, gi[r, c], gv[r, c], wi[r, c], wv[r, c]))


# ---- CPU -----------------------------------------------------------------------------------------------------------------
def test_inorder_reference_on_a_hand_worked_case():
    # dim 3, u = (1, 1, 1): the item rows sum 2^60, 1 and -2^60 in three orders; 2^60 + 1 rounds to 2^60 in float64
    big = 2.0 ** 60
    U = np.ones((1, 3), np.float32)
    V = np.array([[big, 1, -big], [1, big, -big], [big, -big, 1], [-1, -2, 0.5], [1, -2, -4]], np.float32)
    bu, bi, mu = [0.5], [0.25, 0.25, 0.25, 1.5, 0.0], 3.0
    S = inorder_scores(U, V, bu, bi, mu)
    assert S.tolist() == [[3.75, 3.75, 4.75, 2.5, -1.5]]
    # |v|: every row's products are non-negative
    assert inorder_scores(U, V, bu, bi, mu, abs_item=True)[0, 3:].tolist() == [8.5, 10.5]
    # the bias adds in the header's order: (2^53 + 1) + 1 rounds twice to 2^53, 2^53 + (1 + 1) does not
    S = inorder_scores([[2.0 ** 26]], [[2.0 ** 27]], [1.0], [1.0], 0.0)
    assert S[0, 0] == 2.0 ** 53 != 2.0 ** 53 + 2
    # ranking: score descending, lowest id on ties, excluded ids (duplicates) never returned, (-inf, -1) past the end
    S = np.array([[1.0, 3.0, 3.0, np.nan, 2.0, 3.0], [0.0, -0.0, 5.0, 5.0, 0.0, -np.inf]])
    idx, val = ref_rank(S, 5, [[2, 2, 0], [3]])
    assert idx.tolist() == [[1, 5, 4, -1, -1], [2, 0, 1, 4, 5]]
    assert val[0].tolist() == [3.0, 3.0, 2.0, -np.inf, -np.inf] and val[1].tolist() == [5.0, 0.0, -0.0, 0.0, -np.inf]


def test_inorder_reference_differs_from_the_blas_order():
    """At dim 512 the order of the adds shows: u = 1, v = (2^60, 1, ..., 1, -2^60).  In order, every 1 is lost against
    2^60 and the sum is 0; the exact sum is 510; a BLAS that sums in panels or lanes keeps some of the ones."""
    d = 512
    U = np.ones((2, d), np.float32)
    V = np.ones((3, d), np.float32)
    V[:, 0], V[:, -1] = 2.0 ** 60, -2.0 ** 60
    S = inorder_scores(U, V, np.zeros(2), np.zeros(3), 0.0)
    assert (S == 0.0).all()
    assert math.fsum(np.float64(V[0]) * np.float64(U[0])) == 510.0
    blas = U.astype(np.float64) @ V.astype(np.float64).T
    assert not np.array_equal(S, blas), blas
    # random full-mantissa operands: the two orders disagree in many entries; both stay close to each other
    rng = np.random.default_rng(3)
    U, V = rng.standard_normal((20, d)).astype(np.float32), rng.standard_normal((300, d)).astype(np.float32)
    S = inorder_scores(U, V, np.zeros(20), np.zeros(300), 0.0)
    blas = U.astype(np.float64) @ V.astype(np.float64).T
    assert (S != blas).mean() > 0.1
    np.testing.assert_allclose(S, blas, rtol=1e-12, atol=1e-12)


def test_chunk_and_pass_mirror_and_what_the_sweeps_reach():
    L = _lib.load()
    calls = sweep_calls()
    for n, I, k, _ in calls:
        assert L.tfr_rank_users_workspace_bytes(n, I, k) == ru_workspace(n, I, k), (n, I, k)
    for n, I, k in ((4096, 62423, 50), (1, 1, 1), (70000, 1000, 1024), (3, (1 << 31) - 1, 7)):
        assert L.tfr_rank_users_workspace_bytes(n, I, k) == ru_workspace(n, I, k), (n, I, k)
    # the knob: rounded up to a multiple of 1024, clamped to [1024, 16384]
    assert [ru_chunk_items(c) for c in KNOBS] == [1024, 3072, 16384, 16384, 1024, 1024]
    assert ru_chunk_items(RANK_CHUNK_DEFAULT) == RANK_CHUNK_DEFAULT and RU_MAX_K == 1024
    # the ML-25M shape: a pass holds about 2150 queries
    assert ru_pass_queries(10 ** 6, 62423) == 2150
    passes = chunks = 0
    short_last = False
    k_classes = set()
    for n, I, k, knob in calls:
        chunk = ru_chunk_items(knob)
        nb = ru_pass_queries(n, I)
        passes = max(passes, -(-n // nb))
        chunks = max(chunks, -(-I // chunk))
        short_last |= 0 < I % chunk < k
        k_classes.add(next(c for c in (1, 32, 256, 512, 1024) if k <= c))
    # multi-pass: three passes of 128 queries, the last one partial; the single-pass slices are one pass each
    nb = ru_pass_queries(MP_QUERIES, MP_ITEMS)
    assert nb == 128 and MP_QUERIES > 2 * nb and MP_QUERIES % nb != 0 and passes == 3
    assert all(ru_pass_queries(min(128, MP_QUERIES - s), MP_ITEMS) == min(128, MP_QUERIES - s)
               for s in range(0, MP_QUERIES, 128))
    assert chunks > 2 * 32                       # a merge lane holds three lists
    assert short_last
    assert k_classes == {1, 32, 256, 512, 1024}
    # every item tied, k = 1024 at the default chunk: the first chunk holds more ties at the threshold than k, and k is
    # more than RU_SEL_THREADS of them, taken in id order over several steps of the scan
    assert dict(TIE_CASES)["all"] > RANK_CHUNK_DEFAULT > RU_MAX_K > RU_SEL_THREADS and RU_MAX_K in TIE_KS
    # the scoring dims: one short of, at and one past every 32-dim staging step up to 512, and 1 and 2
    assert {d % 32 for d in DIMS} >= {0, 1, 31} and max(DIMS) == 512 and min(DIMS) == 1


# ---- GPU: helpers ----------------------------------------------------------------------------------------------------------
def _tables(U, I, d, seed):
    """fp32 features with exponents spread over 2^-6 .. 2^2 (summation order shows in the low bits), biases and mu"""
    rng = np.random.default_rng(seed)
    feat = lambda n: (rng.standard_normal((n, d)) * 2.0 ** rng.integers(-6, 3, (n, d))).astype(np.float32)
    return dict(mu=np.array([rng.standard_normal()], np.float32),
                user_bias=rng.standard_normal(U).astype(np.float32), item_bias=rng.standard_normal(I).astype(np.float32),
                user_feat=feat(U), item_feat=feat(I))


LAYOUTS = {"adam": _lib.README_FLAGS, "sgd": _lib.OPT_SGD, "fork": _lib.FORK_FLAGS}


def _engine(tabs, layout="adam"):
    from tf_recomm_b200.engine import SvdEngine
    U, d = tabs["user_feat"].shape
    eng = SvdEngine(U, tabs["item_feat"].shape[0], d, 1e-3, 0.05, flags=LAYOUTS[layout], tables=tabs)
    assert eng.feat_stride == (0 if eng.sgd else 3 * d)
    return eng


def _scores(tabs, q, abs_item=False):
    return inorder_scores(tabs["user_feat"][q], tabs["item_feat"], tabs["user_bias"][q], tabs["item_bias"],
                          tabs["mu"][0], abs_item)


def _exclusions(U, I, k, seed, edges=True):
    """Per-user excluded ids, ascending with duplicates: user 0 every item, user 1 all but fewer than k, the last user
    nothing, every other user random ids plus some of the ids on the 1024-item chunk edges."""
    rng = np.random.default_rng(seed)
    lists = []
    edge_ids = np.array([i for c in range(RU_MIN_CHUNK, I + 1, RU_MIN_CHUNK) for i in (c - 1, c) if i < I] + [0, I - 1])
    for u in range(U):
        if u == 0:
            ids = np.arange(I)
        elif u == 1:
            ids = rng.permutation(I)[:I - min(max(k // 2, k - 3), I)]
        elif u == U - 1:
            ids = np.zeros(0, np.int64)
        else:
            ids = rng.integers(0, I, rng.integers(0, min(I // 8, 3000) + 2))
            if edges:
                ids = np.concatenate([ids, edge_ids[rng.random(len(edge_ids)) < 0.5]])
        ids = np.sort(np.concatenate([ids, ids[:: 3]])).astype(np.int32)
        lists.append(ids)
    return lists


def _queries(U, n, seed):
    """n query ids, shuffled, with duplicates, users 0, 1 and U - 1 in it"""
    rng = np.random.default_rng(seed)
    q = np.concatenate([[0, 1, U - 1, 1], rng.integers(0, U, n - 4)]).astype(np.int32)
    return q[rng.permutation(n)]


@pytest.fixture
def rank_chunk():
    """Sets the RANK_CHUNK knob for a test and restores it afterwards."""
    old = _lib.tune_get("RANK_CHUNK")
    yield lambda v: _lib.tune_set("RANK_CHUNK", v)
    _lib.tune_set("RANK_CHUNK", old)


def _c_rank(eng, q, k, excl=None):
    """tfr_rank_users straight from the C ABI (k not clamped); excl: per-user id lists (as _exclusions) or None."""
    import torch
    dev = eng.device
    q = np.asarray(q, np.int32)
    n = len(q)
    q_dev = torch.from_numpy(q).to(dev)
    idx = torch.empty(n, k, dtype=torch.int32, device=dev)
    val = torch.empty(n, k, dtype=torch.float64, device=dev)
    nbytes = _lib.check(eng.L.tfr_rank_users_workspace_bytes(n, eng.I, k))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    indptr = items = None
    if excl is not None:
        indptr = torch.from_numpy(np.concatenate([[0], np.cumsum([len(x) for x in excl])]).astype(np.int64)).to(dev)
        items = torch.from_numpy(np.concatenate(excl).astype(np.int32)).to(dev)
    T = eng.t
    with torch.cuda.device(dev):
        _lib.check(eng.L.tfr_rank_users(T["user_feat"].data_ptr(), T["item_feat"].data_ptr(), T["user_bias"].data_ptr(),
                                        T["item_bias"].data_ptr(), T["mu"].data_ptr(), eng.U, eng.I, eng.d,
                                        eng.feat_stride, eng.feat_stride, eng.flags & _lib.ABS_ITEM, q_dev.data_ptr(), n,
                                        k, indptr.data_ptr() if excl is not None else None,
                                        items.data_ptr() if excl is not None else None, val.data_ptr(), idx.data_ptr(),
                                        ws.data_ptr(), nbytes, torch.cuda.current_stream(dev).cuda_stream))
    return idx.cpu().numpy(), val.cpu().numpy()


def _pair_csr(excl):
    import torch
    from tf_recomm_b200.engine import PairCSR
    indptr = np.concatenate([[0], np.cumsum([len(x) for x in excl])]).astype(np.int64)
    return PairCSR(torch.from_numpy(indptr).cuda(), torch.from_numpy(np.concatenate(excl).astype(np.int32)).cuda())


# ---- GPU: tfr_rank_users ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("layout,d", [("adam", d) for d in DIMS] + [("sgd", d) for d in DIMS] +
                         [("fork", d) for d in FORK_DIMS])
def test_rank_users_at_every_dim_class(rank_chunk, layout, d):
    """Every 32-dim staging step of the score kernel, on the interleaved Adam table (stride 3 * dim), the SGD table
    (stride dim) and the fork model's u.|v|; through the engine without exclusions and the C ABI with them."""
    I, U = dim_items(d), 60
    tabs = _tables(U, I, d, seed=d)
    eng = _engine(tabs, layout)
    q = _queries(U, DIM_QUERIES, seed=d)
    excl = _exclusions(U, I, DIM_K, seed=d)
    S = _scores(tabs, q, abs_item=layout == "fork")
    want, want_x = ref_rank(S, DIM_K), ref_rank(S, DIM_K, [excl[u] for u in q])
    for chunk in CHUNKS:
        rank_chunk(chunk)
        assert_same(eng.rank_users(q, k=DIM_K), want, "chunk %d" % chunk)
        assert_same(_c_rank(eng, q, DIM_K, excl), want_x, "chunk %d, excluded" % chunk)


@pytest.mark.gpu
@pytest.mark.parametrize("k", KS)
@pytest.mark.parametrize("masked", [False, True])
def test_rank_users_at_every_k_class(rank_chunk, k, masked):
    """k on each side of the warp, the 256-thread select loops and the bitonic padding up to 1024; at chunk 1024 the last
    chunk (952 items) is shorter than k >= 953.  User 0 has every item excluded, user 1 fewer than k rankable ones."""
    U = 60
    tabs = _tables(U, K_ITEMS, K_DIM, seed=k)
    eng = _engine(tabs)
    q = _queries(U, K_QUERIES, seed=k)
    excl = _exclusions(U, K_ITEMS, k, seed=k) if masked else None
    want = ref_rank(_scores(tabs, q), k, [excl[u] for u in q] if masked else None)
    if masked:
        assert (want[0][q == 0] == -1).all() and (want[0][q == 1][:, -1] == -1).all()
    for chunk in CHUNKS:
        rank_chunk(chunk)
        assert_same(_c_rank(eng, q, k, excl), want, "chunk %d" % chunk)


@pytest.mark.gpu
@pytest.mark.parametrize("I", ITEM_COUNTS)
def test_rank_users_at_the_chunk_edges(rank_chunk, I):
    U, d = 50, 24
    tabs = _tables(U, I, d, seed=I)
    eng = _engine(tabs)
    q = _queries(U, _item_queries(I), seed=I)
    S = _scores(tabs, q)
    for k in ITEM_KS:
        excl = _exclusions(U, I, k, seed=k)
        want = ref_rank(S, k, [excl[u] for u in q])
        for chunk in CHUNKS:
            rank_chunk(chunk)
            assert_same(_c_rank(eng, q, k, excl), want, "k %d chunk %d" % (k, chunk))


@pytest.mark.gpu
@pytest.mark.parametrize("I", FEW_ITEMS)
def test_rank_users_with_fewer_items_than_k(rank_chunk, I):
    """k > n_items through the C ABI (the engine clamps k; the ABI ranks every item and pads the rest)."""
    U = 20
    tabs = _tables(U, I, 9, seed=I)
    eng = _engine(tabs)
    q = _queries(U, 20, seed=I)
    S = _scores(tabs, q)
    for k in (I + 1, RU_MAX_K):
        excl = _exclusions(U, I, k, seed=I)
        want, want_x = ref_rank(S, k), ref_rank(S, k, [excl[u] for u in q])
        assert (want[0][:, I:] == -1).all()
        for chunk in CHUNKS:
            rank_chunk(chunk)
            assert_same(_c_rank(eng, q, k), want, "k %d chunk %d" % (k, chunk))
            assert_same(_c_rank(eng, q, k, excl), want_x, "k %d chunk %d, excluded" % (k, chunk))


def _tied_tables(name, U, I, seed):
    tabs = _tables(U, I, 16, seed)
    V, b = tabs["item_feat"], tabs["item_bias"]
    if name == "all":                 # every item the same row: every score of a user ties
        V[:], b[:] = V[0], b[0]
    elif name == "straddle":          # groups i % 700 (members 700 apart) and the run 1016 .. 1031 across the 1024 edge
        src = np.arange(I) % 700
        src[1016:1032] = 1016
        V[:], b[:] = V[src], b[src]
        b[src == 1016] += 1000.0      # the run ranks first
    elif name == "flat_chunk":        # items 1024 .. 2047 (one 1024-item chunk) equal, and best
        V[1024:2048], b[1024:2048] = V[1024], b[1024] + 50.0
    return tabs


@pytest.mark.gpu
@pytest.mark.parametrize("name,I", TIE_CASES)
@pytest.mark.parametrize("k", TIE_KS)
def test_rank_users_ties(rank_chunk, name, I, k):
    """Ties at the radix threshold are taken in id order, 256 positions at a time; tie groups split over chunks are merged
    lowest id first; a chunk whose rankable keys are all equal."""
    U = 40
    tabs = _tied_tables(name, U, I, seed=k)
    eng = _engine(tabs)
    q = _queries(U, 24, seed=k)
    S = _scores(tabs, q)
    excl = _exclusions(U, I, k, seed=k)
    want, want_x = ref_rank(S, k), ref_rank(S, k, [excl[u] for u in q])
    if name == "all":
        assert (want[0] == np.arange(k)).all()
    for chunk in CHUNKS:
        rank_chunk(chunk)
        assert_same(_c_rank(eng, q, k), want, "chunk %d" % chunk)
        assert_same(_c_rank(eng, q, k, excl), want_x, "chunk %d, excluded" % chunk)


@pytest.mark.gpu
def test_rank_chunk_knob(rank_chunk):
    """RANK_CHUNK 1024, 3000 (-> 3072), 16384 and values out of range (clamped): the same bits as the reference."""
    U = 30
    tabs = _tables(U, KNOB_ITEMS, 20, seed=5)
    eng = _engine(tabs)
    q = _queries(U, 16, seed=5)
    excl = _exclusions(U, KNOB_ITEMS, KNOB_K, seed=5)
    want = ref_rank(_scores(tabs, q), KNOB_K, [excl[u] for u in q])
    for chunk in KNOBS:
        rank_chunk(chunk)
        assert_same(_c_rank(eng, q, KNOB_K, excl), want, "RANK_CHUNK %d" % chunk)


@pytest.mark.gpu
@pytest.mark.parametrize("I", MERGE_ITEMS)
@pytest.mark.parametrize("k", MERGE_KS)
def test_merge_of_more_than_32_lists(rank_chunk, I, k):
    """41 and 68 chunks of 1024 items: merge lanes hold two and three lists."""
    U = 12
    tabs = _tables(U, I, 12, seed=I + k)
    eng = _engine(tabs)
    q = _queries(U, 8, seed=k)
    excl = _exclusions(U, I, k, seed=k)
    rank_chunk(1024)
    assert_same(_c_rank(eng, q, k, excl), ref_rank(_scores(tabs, q), k, [excl[u] for u in q]))
    assert_same(_c_rank(eng, q, k), ref_rank(_scores(tabs, q), k))


@pytest.mark.gpu
def test_rank_users_in_several_passes(rank_chunk):
    """2^20 items: a pass holds 128 queries, 300 queries take three passes, the last one partial.  The whole call equals
    single-pass calls on slices of 128 queries, and the rows at each pass edge equal the reference (computed row by row:
    the whole float64 matrix would take 2.4 GB)."""
    U = 400
    tabs = _tables(U, MP_ITEMS, MP_DIM, seed=11)
    eng = _engine(tabs)
    q = np.random.default_rng(11).permutation(U)[:MP_QUERIES].astype(np.int32)
    q[[5, 200]] = 0, 1                     # every item excluded / fewer than k rankable, in two passes
    excl = _exclusions(U, MP_ITEMS, MP_K, seed=11, edges=False)
    for chunk in CHUNKS:
        rank_chunk(chunk)
        whole = _c_rank(eng, q, MP_K, excl)
        if chunk == RANK_CHUNK_DEFAULT:
            parts = [_c_rank(eng, q[s:s + 128], MP_K, excl) for s in range(0, MP_QUERIES, 128)]
            assert_same(whole, tuple(np.concatenate(x) for x in zip(*parts)), "slices")
        for r in (0, 5, 127, 128, 200, 255, 256, MP_QUERIES - 1):
            want = ref_rank(_scores(tabs, q[[r]]), MP_K, [excl[q[r]]])
            assert_same((whole[0][[r]], whole[1][[r]]), want, "chunk %d, row %d" % (chunk, r))


# ---- GPU: the exact paths of rank_all_users -----------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("d", [1, 31, 33, 65, 127, 129, 255, 257, 511, 512])
@pytest.mark.parametrize("I", [1023, 1024, 1025, 2049])
@pytest.mark.parametrize("masked", [False, True])
def test_allpairs_exact_rows(d, I, masked):
    """Dims the tensor cores cannot take send every row through allpairs_exact_rows_kernel (one 1024-thread CTA per row)."""
    U = 24
    tabs = _tables(U, I, d, seed=d + I)
    eng = _engine(tabs)
    excl = _exclusions(U, I, 128, seed=d) if masked else None
    S = _scores(tabs, np.arange(U))
    for k in (1, 37, AP_MAX_CAND):
        idx, val, n_unc = eng._rank_excluding(k, None, _pair_csr(excl) if masked else None)
        assert n_unc == U
        assert_same((idx, val), ref_rank(S, k, excl), "k %d" % k)


def _rescore_tables(U, I, d, seed):
    """Well-separated scores (feature products small next to the spread of the item biases), so that most rows are
    certified by allpairs_rescore_kernel and do not take the exact path."""
    rng = np.random.default_rng(seed)
    return dict(mu=np.array([0.5], np.float32), user_bias=rng.standard_normal(U).astype(np.float32),
                item_bias=(4 * rng.standard_normal(I)).astype(np.float32),
                user_feat=(0.1 * rng.standard_normal((U, d))).astype(np.float32),
                item_feat=(0.1 * rng.standard_normal((I, d))).astype(np.float32))


@pytest.mark.gpu
@pytest.mark.parametrize("d", [32, 64, 96, 128])
@pytest.mark.parametrize("k,n_cand", [(1, 1), (5, 8), (10, 10), (10, 24), (50, 64), (100, 128), (128, 128)])
def test_allpairs_rescore_in_bits(d, k, n_cand):
    """The float64 values of the tensor-core ranking (candidates rescored by allpairs_rescore_kernel), without and with an
    exclusion list: ids and bits equal the in-order reference, n_cand below 11 (a buffer of 11) and 128 included."""
    U, I = 200, 2500
    tabs = _rescore_tables(U, I, d, seed=d + k)
    eng = _engine(tabs)
    S = _scores(tabs, np.arange(U))
    excl = _exclusions(U, I, k, seed=d, edges=False)
    idx, val, n_unc = eng.rank_all_users(k=k, n_cand=n_cand)
    assert_same((idx, val), ref_rank(S, k), "all items")
    idx, val, n_unc_x = eng._rank_excluding(k, n_cand, _pair_csr(excl))
    assert_same((idx, val), ref_rank(S, k, excl), "excluded")
    if n_cand >= k + 10:
        assert n_unc < U // 2 and n_unc_x < U // 2, (n_unc, n_unc_x)


# ---- GPU: tfr_topk_rows on given fp32 matrices --------------------------------------------------------------------------
def _topk_matrix(n_cols, seed):
    """Rows: random; random with NaN and +-inf; a few values (exact ties) and +-0; all equal; all NaN; NaN with a few
    -inf; only infinities."""
    rng = np.random.default_rng(seed)
    rows = [rng.standard_normal(n_cols)]
    r = rng.standard_normal(n_cols)
    r[rng.random(n_cols) < 0.2] = np.nan
    r[rng.random(n_cols) < 0.05] = np.inf
    r[rng.random(n_cols) < 0.05] = -np.inf
    rows.append(r)
    r = rng.integers(-3, 4, n_cols) * 0.25
    r[rng.random(n_cols) < 0.3] = -0.0
    rows.append(r)
    rows.append(np.full(n_cols, 1.5))
    rows.append(np.full(n_cols, np.nan))
    r = np.full(n_cols, np.nan)
    r[rng.random(n_cols) < 0.1] = -np.inf
    rows.append(r)
    rows.append(np.where(rng.random(n_cols) < 0.5, np.inf, -np.inf))
    return np.array(rows, np.float32)


@pytest.mark.gpu
@pytest.mark.parametrize("n_cols", [1, 31, 1023, 1024, 1025, 5000])
def test_topk_rows(n_cols):
    """Pure selection, so the reference is exact: lexsort of the given scores, NaN never ranked, -1 past the rankable
    ones; rows at a stride past n_cols whose padding (+inf) must never be read."""
    import torch
    L = _lib.load()
    M = _topk_matrix(n_cols, seed=n_cols)
    n_rows, stride = M.shape[0], n_cols + 13
    padded = np.full((n_rows, stride), np.inf, np.float32)
    padded[:, :n_cols] = M
    dev = torch.device("cuda")
    src = torch.from_numpy(padded).to(dev)
    for k in sorted({1, 33, RU_MAX_K, n_cols + 1}):
        val = torch.empty(n_rows, k, dtype=torch.float32, device=dev)
        idx = torch.empty(n_rows, k, dtype=torch.int32, device=dev)
        _lib.check(L.tfr_topk_rows(src.data_ptr(), n_rows, n_cols, stride, k, val.data_ptr(), idx.data_ptr(),
                                   torch.cuda.current_stream().cuda_stream))
        assert_same((idx, val), ref_rank(M, k), "k %d" % k)
