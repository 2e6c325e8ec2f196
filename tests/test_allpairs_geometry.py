"""The tcgen05 all-pairs sweep (allpairs_tc_kernel<KCHUNKS, TOPK, OBS, EXCL> in csrc/allpairs.cu) at every tile, stride,
consumer and compaction edge, bit for bit against float64.

A CTA owns AP_BM = 128 user rows and sweeps the item table in tiles of AP_BN = 128 items, dim in KCHUNKS = dim / AP_KC
chunks of 32.  Two epilogue warps share each 32-row quarter and split a tile's columns in halves of 64; a lane keeps
four arg-max chains (column % 4) for the top-1, one unsorted candidate buffer of C = 4K entries per row-half for the
top-k (K = max(n_cand, 11), compacted by a warp radix select whenever fewer than 32 slots are left after a 32-column
chunk), and walks the row's CSR lists of observed pairs (OBS) and excluded items (EXCL), skipping the other half's
columns at each tile start.

The inputs make every output exact, so nothing is compared within a tolerance:
  * features are small integers times 2^e (at most 11 significant bits: tf32 reads them as they are), biases and mu are
    on the grid of the products, and every partial sum of a score stays below 2^23 grid steps.  The tensor cores' fp32
    dot product is then exact in any accumulation order, and s = fl(fl(D + b_u) + fl(b_i + mu)) is the float64 score;
  * ratings are on the same grid, so (s - r)^2 and its sums are exact in float64;
  * the top-k runs with AP_STAGES = 3 (sweep and rescore, no exact fallback) on these inputs: a rescored candidate
    set ranks exactly only if the buffers kept every row's true top k, so a lost candidate shows instead of being
    repaired by the fallback;
  * the well-separated tables (candidate buffers, exclusion walk) put a gap larger than the certificate's E_u between
    consecutive exact scores of every row's top k + 1 rankable items: every row must certify.
"""
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


AP_BM = _constant("allpairs.cu", "AP_BM")
AP_BN = _constant("allpairs.cu", "AP_BN")
AP_KC = _constant("allpairs.cu", "AP_KC")
AP_MAX_CAND = _constant("allpairs.cu", "AP_MAX_CAND")
assert re.search(r"constexpr int AP_EPL = 4 \* AP_MAX_CAND / 32;", _source("allpairs.cu"))
AP_EPL = 4 * AP_MAX_CAND // 32
_floor = re.search(r"static int ap_buffer_k\(int n_cand\) \{ return n_cand > (\d+) \? n_cand : (\d+); \}",
                   _source("allpairs.cu"))
assert _floor and _floor.group(1) == _floor.group(2)
BUF_FLOOR = int(_floor.group(1))
HALF = AP_BN // 2


def buffer_k(n_cand):
    """allpairs.cu ap_buffer_k: entries a row-half keeps after a compaction"""
    return max(n_cand, BUF_FLOOR)


# ---- the sweeps (the GPU tests run exactly these; the CPU tests check what they reach) ----------------------------------
DIMS = [32, 64, 96, 128]
ITEMS = [1, 2, 63, 64, 65, 127, 128, 129, 191, 192, 193, 255, 256, 257, 2000]
USERS = [1, 31, 32, 33, 127, 128, 129, 255, 256, 257]
GRID_U, GRID_I = 129, 193                   # the partner of each line of the grid: both tiles partial
EXTRA_SHAPES = [(1, 1), (256, 128), (128, 63), (33, 2000)]
WAVE_EXTRA, WAVE_I = 77, 65                 # U = 128 * SMs + 77: more than one wave of CTAs
STRIDES = {"adam": (3, 3), "sgd": (1, 1), "mixed": (3, 1)}   # (user, item) row stride in units of dim
GRID_K, GRID_CAND = 10, 24


def grid_shapes():
    shapes = [(GRID_U, I) for I in ITEMS] + [(U, GRID_I) for U in USERS if U != GRID_U] + EXTRA_SHAPES
    return list(dict.fromkeys(shapes))


PATTERNS = ["ascending", "descending", "saw32", "saw64", "saw128", "random"]
PAIRS = [(1, 1), (5, 5), (3, 8), (10, 24), (50, 64), (127, AP_MAX_CAND)]   # (k, n_cand)
SEP_U, SEP_I = 257, 2000
TOP_RANKS, TOP_GAP = 160, 12                # the best 160 keys of a row are 12 apart (E_u < 8 at these inputs)
EXCL_PATTERNS = ["ascending", "saw64", "random"]
EXCL_ITEMS = [2000, 257]
EXCL_EDGES = (0, 63, 64, 65, 127, 128, 129)
TIE_GROUP = (7, 9, 64, 66, 130, 195)        # identical item rows: chains 3, 1, 0, 2, 2, 3; halves 0, 0, 1, 1, 0, 1


# ---- exact inputs -----------------------------------------------------------------------------------------------------
def _grid(rng, shape, lo, hi, e):
    """integers in [lo, hi] times 2^e, as float32 (exact)"""
    return (rng.integers(lo, hi + 1, shape) * 2.0 ** e).astype(np.float32)


def _tables(mu, ub, ib, uf, vf):
    return dict(mu=np.array([mu], np.float32), user_bias=np.asarray(ub, np.float32), item_bias=np.asarray(ib, np.float32),
                user_feat=np.ascontiguousarray(uf, np.float32), item_feat=np.ascontiguousarray(vf, np.float32))


def tie_rows(U):
    return np.arange(U) % 5 == 2


def flat_rows(U):
    f = np.zeros(U, bool)
    f[[0, U - 1]] = True
    f[tie_rows(U)] = False
    return f


def grid_tables(U, I, d, seed):
    """Features in {-8..8} * 2^-3 (products on 2^-6), biases and mu on 2^-6, item bias b_i = -v_i[1].  Rows u % 5 == 2
    are e_0 and score v_i[0] - v_i[1] + b_u + mu: only the identical rows of TIE_GROUP (v[0] = 1, v[1] = -1) reach its
    maximum, 2.  Rows 0 and U - 1 (unless tie rows) are e_1: every score of theirs is b_u + mu."""
    rng = np.random.default_rng(seed)
    uf, vf = _grid(rng, (U, d), -8, 8, -3), _grid(rng, (I, d), -8, 8, -3)
    vf[:, 0] = _grid(rng, I, -8, 7, -3)
    ib = (0.0 - vf[:, 1]).astype(np.float32)   # 0.0 - x: no -0.0
    tie = [i for i in TIE_GROUP if i < I]
    if tie:
        vf[tie] = vf[tie[0]]
        vf[tie, 0], vf[tie, 1], ib[tie] = 1.0, -1.0, 1.0
    t, f = tie_rows(U), flat_rows(U)
    uf[t] = 0.0
    uf[t, 0] = 1.0
    uf[f] = 0.0
    uf[f, 1] = 1.0
    return _tables(3.0, _grid(rng, U, -64, 64, -6), ib, uf, vf)


def pattern_ranks(pattern, I, seed=0):
    """rank (0 = worst) of each item id in the row order of the pattern"""
    i = np.arange(I)
    if pattern == "ascending":
        key = i
    elif pattern == "descending":
        key = -i
    elif pattern.startswith("saw"):
        P = int(pattern[3:])
        key = (i % P) * I + i // P              # rising inside each period of P ids; the peaks rise period by period
    elif pattern == "random":
        key = np.random.default_rng(seed).permutation(I)
    else:
        raise ValueError(pattern)
    return np.argsort(np.argsort(key, kind="stable"), kind="stable")


def key_values(r, I):
    """Ranks -> exact keys: the ranks below the best TOP_RANKS are the keys 0, 1, ...; the best TOP_RANKS are TOP_GAP
    apart above them, multiples of 4 below 4096 (at most 10 significant bits)."""
    n_dense = max(I - TOP_RANKS, 0)
    base = -(-n_dense // 4) * 4 + TOP_GAP
    return np.where(r < n_dense, r, base + TOP_GAP * (r - n_dense)).astype(np.float64)


def separated_tables(U, I, d, pattern, seed):
    """u = (1, noise), v = (key, noise): noise in {-1, 0, 1} * 2^-5 (products on 2^-10), biases in {-32..32} * 2^-10,
    mu = 0.5.  The exact scores follow the pattern's keys to within 0.2; the best TOP_RANKS are TOP_GAP apart."""
    rng = np.random.default_rng(seed)
    uf, vf = _grid(rng, (U, d), -1, 1, -5), _grid(rng, (I, d), -1, 1, -5)
    uf[:, 0] = 1.0
    vf[:, 0] = key_values(pattern_ranks(pattern, I, seed), I)
    return _tables(0.5, _grid(rng, U, -32, 32, -10), _grid(rng, I, -32, 32, -10), uf, vf)


def tied_tables(U, I, d, order, seed):
    """Items in groups of 50 identical rows (features and bias), group keys ascending or descending with the id: every
    row's scores tie in runs of 50 ids, so compactions meet exact ties at their threshold."""
    t = separated_tables(U, I, d, "ascending", seed)
    g = np.arange(I) // 50
    src = g * 50
    t["item_feat"] = np.ascontiguousarray(t["item_feat"][src])
    t["item_bias"] = np.ascontiguousarray(t["item_bias"][src])
    t["item_feat"][:, 0] = (g if order == "ascending" else g.max() - g) * 4.0
    return t


def model_tables(t, abs_item):
    return dict(t, item_feat=np.abs(t["item_feat"])) if abs_item else t


def exact_scores(t):
    """The float64 score matrix, checked to be exact: a second summation order gives the same bits."""
    U64, V64 = t["user_feat"].astype(np.float64), t["item_feat"].astype(np.float64)
    ub, ib, mu = t["user_bias"].astype(np.float64), t["item_bias"].astype(np.float64), float(t["mu"][0])
    M = ((U64 @ V64.T + ub[:, None]) + ib[None, :]) + mu
    M2 = (V64[:, ::-1] @ U64[:, ::-1].T).T + (ub[:, None] + (ib[None, :] + mu))
    assert np.array_equal(M, M2), "inputs not exact in float64"
    return M


def _pow2_step(x):
    """the largest 2^e (e >= -60) that every value of x is a multiple of"""
    x = np.asarray(x, np.float64)
    return next(2.0 ** e for e in range(20, -61, -1) if not np.mod(x, 2.0 ** e).any())


def grid_step(t):
    """the grid of the scores: a step that every product, bias and mu is a multiple of"""
    return min(_pow2_step(t["user_feat"]) * _pow2_step(t["item_feat"]), _pow2_step(t["user_bias"]),
               _pow2_step(t["item_bias"]), _pow2_step(t["mu"]))


def is_tf32(x):
    return not (np.ascontiguousarray(x, np.float32).view(np.uint32) & np.uint32(0x1FFF)).any()


def cert_bound(t):
    """E_u of allpairs_rescore_kernel, per user: (2^-9 + dim 2^-22) ||u|| V + 2^-22 (||u|| V + |b_u| + B)"""
    d = t["user_feat"].shape[1]
    V = np.sqrt((t["item_feat"].astype(np.float64) ** 2).sum(axis=1)).max()
    B = float(np.abs(t["item_bias"] + t["mu"][0]).max())
    uv = np.sqrt((t["user_feat"].astype(np.float64) ** 2).sum(axis=1)) * V
    return (2.0 ** -9 + d * 2.0 ** -22) * uv + 2.0 ** -22 * (uv + np.abs(t["user_bias"].astype(np.float64)) + B)


def ref_rank(S, k, excluded=None):
    """Every row of S ranked (score descending, lowest id on ties), excluded[r] removed, padded with (-inf, -1)."""
    n, I = S.shape
    idx = np.full((n, k), -1, np.int32)
    val = np.full((n, k), -np.inf)
    for r in range(n):
        cand = np.arange(I)
        if excluded is not None and len(excluded[r]):
            keep = np.ones(I, bool)
            keep[np.asarray(excluded[r], np.int64)] = False
            cand = cand[keep]
        order = cand[np.lexsort((cand, -S[r, cand]))][:k]
        idx[r, :len(order)], val[r, :len(order)] = order, S[r, order]
    return idx, val


def _edges(I):
    """the half and tile edges inside [1, I): multiples of 64"""
    return list(range(HALF, I, HALF))


def obs_lists(U, I, seed):
    """Observed item ids per user (ascending, duplicates adjacent): rows u % 7 == 3 have none (the last row always has
    some); u % 7 == 4 only ids in half-1 columns, u % 7 == 5 only half-0 ids; every other row a few random ids and a
    duplicated run e - 2 .. e + 1 across one half or tile edge e (the edges taken in turn)."""
    rng = np.random.default_rng(seed)
    edges = _edges(I)
    lists = []
    for u in range(U):
        cls = u % 7
        if cls == 3 and u != U - 1:
            ids = np.zeros(0, np.int64)
        elif cls in (4, 5):
            cols = np.arange(I)
            cols = cols[(cols % AP_BN >= HALF) == (cls == 4)]
            ids = rng.choice(cols, min(len(cols), 6)) if len(cols) else np.zeros(0, np.int64)
        else:
            ids = rng.integers(0, I, 5)
            if edges:
                e = edges[u % len(edges)]
                run = np.array([e - 2, e - 1, e - 1, e, e, e + 1])
                ids = np.concatenate([ids, run[(run >= 0) & (run < I)]])
            ids = np.concatenate([ids, ids[::3]])
        lists.append(np.sort(ids).astype(np.int32))
    return lists


def excl_lists(S, k, seed):
    """Excluded item ids per user (ascending, duplicates): row 0 every item; row 1 all but k - 1; the last row none;
    every other row EXCL_EDGES and I - 1, its three best items, a duplicated run e - 2 .. e + 1 across one half or
    tile edge e (in turn), a few random ids, and every third id twice."""
    U, I = S.shape
    rng = np.random.default_rng(seed)
    edges = _edges(I)
    top3 = ref_rank(S, 3)[0]
    lists = []
    for u in range(U):
        if u == 0:
            ids = np.concatenate([np.arange(I), np.arange(0, I, 7)])
        elif u == 1:
            ids = rng.permutation(I)[:I - (k - 1)]
        elif u == U - 1:
            ids = np.zeros(0, np.int64)
        else:
            ids = np.array([e for e in EXCL_EDGES + (I - 1,) if e < I] + top3[u][top3[u] >= 0].tolist())
            if edges:
                e = edges[u % len(edges)]
                run = np.array([e - 2, e - 1, e - 1, e, e, e + 1])
                ids = np.concatenate([ids, run[(run >= 0) & (run < I)]])
            ids = np.concatenate([ids, rng.integers(0, I, 3)])
        ids = np.sort(np.concatenate([ids, ids[::3]])).astype(np.int32)
        lists.append(ids)
    return lists


def _csr(lists):
    indptr = np.concatenate([[0], np.cumsum([len(x) for x in lists])]).astype(np.int64)
    items = np.concatenate(lists).astype(np.int32) if lists else np.zeros(0, np.int32)
    return indptr, items


def obs_rates(lists, seed):
    rng = np.random.default_rng(seed)
    return [_grid(rng, len(x), -320, 320, -6) for x in lists]


def ref_row_se(S, lists, rates):
    se = np.zeros(S.shape[0])
    for u, (ids, r) in enumerate(zip(lists, rates)):
        se[u] = ((S[u, ids] - r.astype(np.float64)) ** 2).sum()
    return se


def geometry_class(d, U, I):
    """(KCHUNKS, last user tile partial, last item tile partial, half of the last column)"""
    return d // AP_KC, U % AP_BM != 0, I % AP_BN != 0, ((I - 1) % AP_BN) // HALF


# ---- CPU --------------------------------------------------------------------------------------------------------------
def test_constants_read_from_the_source():
    assert (AP_BM, AP_BN, AP_KC, AP_MAX_CAND, AP_EPL, BUF_FLOOR) == (128, 128, 32, 128, 16, 11)
    # the floor is the least K whose buffer of 4K takes the K kept entries and a whole chunk of 32 appends
    assert 4 * BUF_FLOOR >= BUF_FLOOR + 32 and 4 * (BUF_FLOOR - 1) < (BUF_FLOOR - 1) + 32
    assert 4 * buffer_k(AP_MAX_CAND) == 32 * AP_EPL
    assert [buffer_k(n) for n in (1, 10, 11, 24, 128)] == [11, 11, 11, 24, 128]
    # the pairs reach the floor with n_cand < 11, n_cand = k, K = 128 (C = 512) and k = 1
    assert any(n < BUF_FLOOR for _, n in PAIRS) and any(k == n for k, n in PAIRS)
    assert any(buffer_k(n) == AP_MAX_CAND for _, n in PAIRS) and any(k == 1 for k, _ in PAIRS)


def _all_input_sets():
    for d in DIMS:
        for U, I in ((GRID_U, 2000), (257, 257), (1, 1)):
            yield "grid", d, grid_tables(U, I, d, seed=d + I)
        for p in PATTERNS:
            yield p, d, separated_tables(SEP_U, SEP_I, d, p, seed=d)
        for order in ("ascending", "descending"):
            yield "tied", d, tied_tables(64, SEP_I, d, order, seed=d)
        yield "fork", d, model_tables(grid_tables(150, 300, d, seed=d), True)
    yield "fork", 20, model_tables(grid_tables(150, 300, 20, seed=20), True)


def test_inputs_are_exact():
    """The premise of every bit-for-bit check: features are tf32 values, every partial sum of a score is a multiple of
    the grid step below 2^23 steps (exact in fp32 in any order), float64 in two orders gives the same bits, and the
    squared errors of the observed pairs sum exactly."""
    for name, d, t in _all_input_sets():
        assert is_tf32(t["user_feat"]) and is_tf32(t["item_feat"]), name
        S = exact_scores(t)
        step = grid_step(t)
        bound = (np.abs(t["user_feat"].astype(np.float64)) @ np.abs(t["item_feat"].astype(np.float64)).T +
                 np.abs(t["user_bias"].astype(np.float64))[:, None] + np.abs(t["item_bias"].astype(np.float64))[None, :] +
                 abs(float(t["mu"][0])))
        assert bound.max() < 2.0 ** 23 * step, (name, d, bound.max(), step)
        assert not np.mod(S, step).any(), name
        assert np.array_equal(S.astype(np.float32).astype(np.float64), S), name
        if name == "grid":
            U, I = S.shape
            lists = obs_lists(U, I, seed=d)
            rates = obs_rates(lists, seed=d)
            se = ref_row_se(S, lists, rates)
            se2 = np.array([((S[u, x[::-1]] - r[::-1].astype(np.float64)) ** 2)[::-1].cumsum()[-1] if len(x) else 0.0
                            for u, (x, r) in enumerate(zip(lists, rates))])
            assert np.array_equal(se, se2)
            assert all(np.abs(S[u, x] - r).max(initial=0) < 2.0 ** 20 * 2.0 ** -6 for u, (x, r) in
                       enumerate(zip(lists, rates)))


def test_tie_and_flat_rows():
    """Rows u % 5 == 2 have their maxima on TIE_GROUP (lowest id 7 in chain 3, after id 9 in chain 1; ids in both halves
    and in the second tile); rows 0 and U - 1 score every item alike."""
    assert [i % 4 for i in TIE_GROUP] == [3, 1, 0, 2, 2, 3]
    assert {(i % AP_BN) // HALF for i in TIE_GROUP} == {0, 1} and {i // AP_BN for i in TIE_GROUP} == {0, 1}
    for d in DIMS:
        for U, I in ((GRID_U, 2000), (GRID_U, 129), (33, 10)):
            S = exact_scores(grid_tables(U, I, d, seed=d))
            tie = [i for i in TIE_GROUP if i < I]
            for u in np.nonzero(tie_rows(U))[0]:
                assert set(np.nonzero(S[u] == S[u].max())[0].tolist()) == set(tie), (d, U, I, u)
            for u in np.nonzero(flat_rows(U))[0]:
                assert (S[u] == S[u, 0]).all()


def _certifies(t, S, k, n_cand, excluded=None):
    """Every row certifies whatever the item order: its k + 1 best rankable exact scores are more than E_u apart (the
    sweep's scores are exact, so the buffers' thresholds are at most the (k + 1)-th best when K > k), or it has too few
    rankable items for a buffer to ever compact (threshold -inf)."""
    E = cert_bound(t)
    K = buffer_k(n_cand)
    assert K > k
    _, val = ref_rank(S, k + 1, excluded)
    for u in range(S.shape[0]):
        rankable = S.shape[1] - (len(set(np.asarray(excluded[u]).tolist())) if excluded is not None else 0)
        if rankable <= 4 * K - 32:
            continue
        if not (np.diff(-val[u]) > E[u]).all():
            return False
    return True


def test_separated_inputs_certify():
    """The premise of n_uncertified == 0: on the well-separated tables the k + 1 best rankable items of every row are
    more than E_u apart, with and without the exclusion lists, and the key layout keeps 10 significant bits."""
    for d in DIMS:
        for p in PATTERNS:
            t = separated_tables(SEP_U, SEP_I, d, p, seed=d)
            S = exact_scores(t)
            assert cert_bound(t).max() < TOP_GAP - 1
            for k, n_cand in PAIRS:
                assert _certifies(t, S, k, n_cand), (d, p, k)
        for p in EXCL_PATTERNS:
            for I in EXCL_ITEMS:
                t = separated_tables(SEP_U, I, d, p, seed=d + I)
                S = exact_scores(t)
                for k, n_cand in PAIRS:
                    assert _certifies(t, S, k, n_cand, excl_lists(S, k, seed=k)), (d, p, I, k)
    # the orders: ascending appends nearly every column, so a row-half at the floor compacts after nearly every chunk
    r = pattern_ranks("saw64", 256)
    assert list(r[:64]) == sorted(r[:64]) and r[63] > r[64]


def _has_run(lists, lo, hi):
    """some list holds every id of [lo, hi], one of them at least twice"""
    for x in lists:
        s = set(x.tolist())
        if all(i in s for i in range(lo, hi + 1)) and len(x) > len(set(x.tolist())) and \
                any((x == i).sum() > 1 for i in range(lo, hi + 1)):
            return True
    return False


def test_the_sweeps_reach_every_geometry_class():
    """The grid reaches every (KCHUNKS, partial user tile, partial item tile, half of the last column) class at every
    stride, and the observed and excluded runs sit on both sides of every half and tile edge, duplicated."""
    want = {(kc, pu, pi, h) for kc in range(1, 5) for pu in (False, True) for pi in (False, True) for h in (0, 1)
            if pi or h == 1}
    got = {geometry_class(d, U, I) for d in DIMS for U, I in grid_shapes()}
    assert got == want
    assert {I for _, I in grid_shapes()} >= set(ITEMS) and {U for U, _ in grid_shapes()} >= set(USERS)
    for U, I in grid_shapes():
        lists = obs_lists(U, I, seed=0)
        assert any(len(x) == 0 for x in lists) or U < 5
        assert len(lists[-1]) > 0
        if I > HALF and U >= 7:
            assert any(len(x) and (x % AP_BN >= HALF).all() for x in lists)
            assert any(len(x) and (x % AP_BN < HALF).all() for x in lists)
    for e in _edges(2000):
        assert _has_run(obs_lists(GRID_U, 2000, seed=0), e - 2, e + 1), e
    S = exact_scores(separated_tables(SEP_U, 2000, 32, "ascending", seed=0))
    for k, _ in PAIRS:
        lists = excl_lists(S, k, seed=k)
        for e in _edges(2000):
            assert _has_run(lists, e - 2, e + 1), (k, e)
        assert len(set(lists[0].tolist())) == 2000 and 2000 - len(set(lists[1].tolist())) == k - 1 and not len(lists[-1])


# ---- GPU: helpers -------------------------------------------------------------------------------------------------------
@pytest.fixture
def ap_stages():
    """Sets the AP_STAGES knob (1 sweep | 2 rescore | 4 exact rows) for a test and restores it afterwards."""
    old = _lib.tune_get("AP_STAGES")
    yield lambda v: _lib.tune_set("AP_STAGES", v)
    _lib.tune_set("AP_STAGES", old)


class Dev:
    """The tables on the device at row strides of us * dim (users) and is_ * dim (items); the floats between rows are
    NaN, which no sweep may read."""

    def __init__(self, t, us=1, is_=1):
        import torch
        self.U, self.d = t["user_feat"].shape
        self.I = t["item_feat"].shape[0]
        self.us, self.is_ = us * self.d, is_ * self.d

        def rows(a, stride):
            x = torch.full((a.shape[0], stride), float("nan"))
            x[:, :self.d] = torch.from_numpy(a)
            return x.cuda()
        self.uf, self.vf = rows(t["user_feat"], self.us), rows(t["item_feat"], self.is_)
        self.ub, self.ib, self.mu = (torch.from_numpy(t[n]).cuda() for n in ("user_bias", "item_bias", "mu"))

    def head(self):
        return (self.uf.data_ptr(), self.vf.data_ptr(), self.ub.data_ptr(), self.ib.data_ptr(), self.mu.data_ptr(),
                self.U, self.I, self.d, self.us, self.is_)


def _stream():
    import torch
    return torch.cuda.current_stream().cuda_stream


def c_allpairs(D, tc):
    """tfr_allpairs -> (scores, best_score, best_item) as numpy"""
    import torch
    L = _lib.load()
    scores = torch.empty(D.U, D.I, dtype=torch.float32, device="cuda")
    bs = torch.empty(D.U, dtype=torch.float32, device="cuda")
    bi = torch.empty(D.U, dtype=torch.int32, device="cuda")
    nbytes = _lib.check(L.tfr_allpairs_workspace_bytes(D.U, D.I, D.d, tc))
    ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    _lib.check(L.tfr_allpairs(*D.head(), tc, scores.data_ptr(), bs.data_ptr(), bi.data_ptr(), ws.data_ptr(), nbytes,
                              _stream()))
    return scores.cpu().numpy(), bs.cpu().numpy(), bi.cpu().numpy()


def _dev_csr(lists, rates=None):
    import torch
    indptr, items = _csr(lists)
    out = [torch.from_numpy(indptr).cuda(), torch.from_numpy(items).cuda()]
    if rates is not None:
        out.append(torch.from_numpy(np.concatenate(rates).astype(np.float32)).cuda())
    return out


def c_consume(D, k, n_cand, obs=None):
    """tfr_allpairs_consume: top-k (k > 0) and / or OBS (obs = device (indptr, items, rates)) in one sweep
    -> (idx, val, n_uncertified, row_se) as numpy (None for what was not asked)"""
    import torch
    L = _lib.load()
    idx = torch.empty(D.U, max(k, 1), dtype=torch.int32, device="cuda")
    val = torch.empty(D.U, max(k, 1), dtype=torch.float64, device="cuda")
    n_unc = torch.zeros(1, dtype=torch.int32, device="cuda")
    row_se = torch.empty(D.U, dtype=torch.float64, device="cuda")
    nbytes = _lib.check(L.tfr_allpairs_topk_workspace_bytes(D.U, D.I, k, n_cand)) if k else 0
    ws = torch.empty(max(nbytes, 1), dtype=torch.uint8, device="cuda")
    o = [x.data_ptr() for x in obs] if obs is not None else [None] * 3
    _lib.check(L.tfr_allpairs_consume(*D.head(), k, n_cand if k else 0, val.data_ptr() if k else None,
                                      idx.data_ptr() if k else None, n_unc.data_ptr() if k else None, *o,
                                      row_se.data_ptr() if obs is not None else None, ws.data_ptr() if k else None,
                                      nbytes, _stream()))
    return (idx.cpu().numpy() if k else None, val.cpu().numpy() if k else None, int(n_unc.item()) if k else None,
            row_se.cpu().numpy() if obs is not None else None)


def c_excluding(D, k, n_cand, lists):
    import torch
    L = _lib.load()
    idx = torch.empty(D.U, k, dtype=torch.int32, device="cuda")
    val = torch.empty(D.U, k, dtype=torch.float64, device="cuda")
    n_unc = torch.zeros(1, dtype=torch.int32, device="cuda")
    nbytes = _lib.check(L.tfr_allpairs_topk_workspace_bytes(D.U, D.I, k, n_cand))
    ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    indptr, items = _dev_csr(lists)
    _lib.check(L.tfr_allpairs_rank_excluding(*D.head(), k, n_cand, indptr.data_ptr(), items.data_ptr(), val.data_ptr(),
                                             idx.data_ptr(), n_unc.data_ptr(), ws.data_ptr(), nbytes, _stream()))
    return idx.cpu().numpy(), val.cpu().numpy(), int(n_unc.item())


def assert_bits(got, want, what=""):
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    g = got.view(np.int64 if got.itemsize == 8 else np.int32)
    w = want.view(np.int64 if want.itemsize == 8 else np.int32)
    bad = np.argwhere(g != w)
    if len(bad):
        raise AssertionError("%s: %d entries differ, first %s: got %r, want %r" % (
            what, len(bad), tuple(bad[0]), got[tuple(bad[0])], want[tuple(bad[0])]))


def assert_ranking(got_idx, got_val, want, what=""):
    assert_bits(got_idx, want[0], what + " ids")
    assert_bits(got_val, want[1], what + " values")


def check_sweep(t, layouts, what):
    """Every consumer of one geometry against float64, at each layout's strides: scores and top-1 on both paths, OBS,
    top-k without the fallback, and top-k + OBS in one sweep equal to the two sweeps apart."""
    U, I = t["user_feat"].shape[0], t["item_feat"].shape[0]
    S = exact_scores(t)
    S32 = S.astype(np.float32)
    k = min(GRID_K, I)
    top = ref_rank(S, k)
    lists = obs_lists(U, I, seed=U + I)
    rates = obs_rates(lists, seed=U + I)
    want_se = ref_row_se(S, lists, rates)
    obs = _dev_csr(lists, rates)
    for layout in layouts:
        D = Dev(t, *STRIDES[layout])
        w = "%s %s" % (what, layout)
        for tc in (1, 0):
            sc, bs, bi = c_allpairs(D, tc)
            assert_bits(sc, S32, "%s tc %d scores" % (w, tc))
            assert_bits(bi, top[0][:, 0], "%s tc %d best_item" % (w, tc))
            assert_bits(bs, top[1][:, 0].astype(np.float32), "%s tc %d best_score" % (w, tc))
        _, _, _, se = c_consume(D, 0, 0, obs)
        assert_bits(se, want_se, w + " row_se")
        idx, val, n_unc, _ = c_consume(D, k, GRID_CAND)
        assert_ranking(idx, val, top, w + " top-k")
        idx2, val2, n_unc2, se2 = c_consume(D, k, GRID_CAND, obs)
        assert_ranking(idx2, val2, (idx, val), w + " top-k with OBS")
        assert_bits(se2, se, w + " row_se with top-k")
        assert n_unc2 == n_unc


# ---- GPU: the geometry grid ----------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("layout", sorted(STRIDES))
@pytest.mark.parametrize("d", DIMS)
def test_sweep_at_every_tile_edge(ap_stages, d, layout):
    ap_stages(3)
    for U, I in grid_shapes():
        check_sweep(grid_tables(U, I, d, seed=d + U + I), [layout], "d %d U %d I %d" % (d, U, I))


@pytest.mark.gpu
@pytest.mark.parametrize("d", DIMS)
def test_sweep_past_one_wave(ap_stages, d):
    ap_stages(3)
    U = AP_BM * _lib.load().tfr_device_sm_count() + WAVE_EXTRA
    check_sweep(grid_tables(U, WAVE_I, d, seed=d), sorted(STRIDES), "d %d U %d I %d" % (d, U, WAVE_I))


# ---- GPU: candidate buffers and compaction -------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("pattern", PATTERNS)
@pytest.mark.parametrize("d", DIMS)
def test_candidate_buffers_keep_the_top_k(d, pattern):
    """Well-separated scores: every row certifies (no fallback), and the ranking is the float64 one in bits, from the
    buffer floor (K = 11, C = 44) to K = 128 (C = 512), in orders that append nearly every column (ascending), almost
    none (descending) or compact at the chunk, half and tile period (sawtooth)."""
    t = separated_tables(SEP_U, SEP_I, d, pattern, seed=d)
    S = exact_scores(t)
    D = Dev(t, *STRIDES[sorted(STRIDES)[PATTERNS.index(pattern) % 3]])
    for k, n_cand in PAIRS:
        idx, val, n_unc, _ = c_consume(D, k, n_cand)
        assert n_unc == 0, (k, n_cand, n_unc)
        assert_ranking(idx, val, ref_rank(S, k), "k %d n_cand %d" % (k, n_cand))


@pytest.mark.gpu
@pytest.mark.parametrize("order", ["ascending", "descending"])
@pytest.mark.parametrize("d", [32, 128])
def test_ties_at_the_compaction_threshold(ap_stages, d, order):
    """Runs of 50 tied ids: a compaction keeps the lowest ids of the ties at its threshold and a later column equal to
    the threshold is dropped.  Without the exact fallback (AP_STAGES = 3) the rescored buffers must still give the
    float64 ranking; with it, the same bits."""
    t = tied_tables(64, SEP_I, d, order, seed=d)
    S = exact_scores(t)
    D = Dev(t, 3, 3)
    for stages in (3, 7):
        ap_stages(stages)
        for k, n_cand in [(5, 5), (10, 24), (50, 64), (127, AP_MAX_CAND)]:
            idx, val, _, _ = c_consume(D, k, n_cand)
            assert_ranking(idx, val, ref_rank(S, k), "stages %d k %d n_cand %d" % (stages, k, n_cand))


# ---- GPU: the exclusion walk ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("I", EXCL_ITEMS)
@pytest.mark.parametrize("pattern", EXCL_PATTERNS)
@pytest.mark.parametrize("d", DIMS)
def test_exclusion_walk(d, pattern, I):
    """Excluded ids on the half and tile edges, duplicated runs across them, the rows' best items, a row with every item
    excluded and one with fewer than k left: every row certifies and ranks its rankable items in float64 bits."""
    t = separated_tables(SEP_U, I, d, pattern, seed=d + I)
    S = exact_scores(t)
    D = Dev(t, *STRIDES[sorted(STRIDES)[DIMS.index(d) % 3]])
    for k, n_cand in PAIRS:
        lists = excl_lists(S, k, seed=k)
        idx, val, n_unc = c_excluding(D, k, n_cand, lists)
        assert n_unc == 0, (k, n_cand, n_unc)
        assert_ranking(idx, val, ref_rank(S, k, lists), "k %d n_cand %d" % (k, n_cand))


# ---- GPU: every all-pairs entry of the engine scores the engine's model ---------------------------------------------------
ENGINE_LAYOUTS = {"readme": _lib.README_FLAGS, "sgd": _lib.OPT_SGD, "fork": _lib.FORK_FLAGS,
                  "fork_adam": _lib.FORK_FLAGS & ~_lib.OPT_SGD}


@pytest.mark.gpu
@pytest.mark.parametrize("d", [32, 128, 20])
@pytest.mark.parametrize("layout", sorted(ENGINE_LAYOUTS))
def test_every_entry_scores_the_engines_model(layout, d):
    """u.|v| + biases under ABS_ITEM, u.v + biases otherwise: rank_all_users with and without exclude (= rank_users of
    every user, bit for bit), allpairs, observed_rmse and ranking_metrics, against float64 of the model's score."""
    from tf_recomm_b200.engine import SvdEngine, TfrError
    flags = ENGINE_LAYOUTS[layout]
    U, I, k = 150, 300, 10
    t = grid_tables(U, I, d, seed=d)
    eng = SvdEngine(U, I, d, 1e-3, 0.05, flags=flags, tables=t)
    S = exact_scores(model_tables(t, bool(flags & _lib.ABS_ITEM)))
    rng = np.random.default_rng(d)
    users, items = rng.integers(0, U, 4 * U).astype(np.int32), rng.integers(0, I, 4 * U).astype(np.int32)
    sets = [np.unique(items[users == u]) for u in range(U)]
    for exclude, want in ((None, ref_rank(S, k)), ((users, items), ref_rank(S, k, sets))):
        what = "exclude" if exclude is not None else "all items"
        idx, val, _ = eng.rank_all_users(k=k, exclude=exclude)
        assert_ranking(idx.cpu().numpy(), val.cpu().numpy(), want, "rank_all_users, " + what)
        q_idx, q_val = eng.rank_users(np.arange(U), k=k, exclude=exclude)
        assert_ranking(q_idx.cpu().numpy(), q_val.cpu().numpy(), want, "rank_users, " + what)
    out = eng.allpairs(want_scores=True)
    assert_bits(out["scores"].cpu().numpy(), S.astype(np.float32), "allpairs scores")
    best = ref_rank(S, 1)
    assert_bits(out["best_item"].cpu().numpy(), best[0][:, 0], "allpairs best_item")
    assert_bits(out["best_score"].cpu().numpy(), best[1][:, 0].astype(np.float32), "allpairs best_score")
    order = np.lexsort((items, users))
    ou, oi = users[order], items[order]
    rates = _grid(rng, len(ou), -320, 320, -6)
    if d % AP_KC == 0 and d <= 4 * AP_KC:
        _, row_se = eng.observed_rmse(ou, oi, rates)
        lists = [oi[ou == u] for u in range(U)]
        assert_bits(row_se.cpu().numpy(), ref_row_se(S, lists, [rates[ou == u] for u in range(U)]), "observed_rmse")
    else:   # the OBS consumer exists only in the tensor-core sweep
        with pytest.raises(TfrError, match="dim % 32 == 0"):
            eng.observed_rmse(ou, oi, rates)
    top = ref_rank(S, k, sets)[0]   # the held-out items: every user's k best unseen ones under the model
    m = eng.ranking_metrics(k, np.repeat(np.arange(U), k), top.reshape(-1), exclude=(users, items))
    assert m["n_users"] == U and m["hr"] == 1.0 and m["precision"] == 1.0 and m["recall"] == 1.0
    assert m["ndcg"] == pytest.approx(1.0, abs=1e-12)
