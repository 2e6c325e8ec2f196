"""The certificate behind every exact all-pairs ranking (allpairs_rescore_kernel): a row's float64-rescored candidates are
its exact top-k when the k-th of them beats T + E_u, T the largest tensor-core score the sweep dropped and E_u a bound on
how far a tensor-core score can be from the exact one.  The inputs here make that inequality tight:

  (a) zero user rows (next to ordinary rows in one 128-row CTA), b_i = i * 2^-35, mu = 3: every item ties in fp32, all
      differ in float64;
  (b) tiny user rows (||u|| ~ 2^-20): the scores sit within an fp32 ulp of mu;
  (c) an all-zero item table (max ||v|| = 0) with the biases of (a);
  (d) tf32 inverts the order: u = s * (1, ..., 1), item components 1 + j * 2^-23 that tf32 reads as 1.0, the best items
      at the highest ids (the lowest-id tie rule keeps the wrong ones);
  (e) near-tie clusters deeper than the candidate buffers, across the column halves and item tiles;
  (f) large biases and mu (10^3 - 10^4) with O(1) features, scores rising with the item id;
  (g) (a), (d), (e) with each row's true top items excluded, and a row whose rankable count lies between k and n_cand.

Every input is a small integer times a power of two, so every float64 score is exact whatever order a sum takes, and the
reference ranking (score descending, lowest id on ties) is unambiguous."""
import numpy as np
import pytest

U_ROWS = 300                      # three 128-row CTAs, the last one partial
DIMS = [32, 64, 96, 128]          # the tcgen05 sweep's dims


# ---- inputs -----------------------------------------------------------------------------------------------------------
def _grid(rng, shape, lo, hi, e):
    """integers in [lo, hi] times 2^e, as float32 (exact)"""
    return (rng.integers(lo, hi + 1, shape) * 2.0 ** e).astype(np.float32)


def _tables(mu, ub, ib, uf, vf):
    return dict(mu=np.array([mu], np.float32), user_bias=np.asarray(ub, np.float32), item_bias=np.asarray(ib, np.float32),
                user_feat=np.ascontiguousarray(uf, np.float32), item_feat=np.ascontiguousarray(vf, np.float32))


def _zero_rows(U):
    z = np.zeros(U, bool)
    z[0:128:3] = True             # every third row of the first CTA, between ordinary rows
    z[[130, 255, U - 1]] = True
    return z


E_CLUSTER = (40, 2200)            # family (e): ids of the near-tie cluster (both column halves of 17 tiles)


def family(name, d, seed=0):
    """-> (tables, rows that must take the exact fallback when nothing is excluded)"""
    rng = np.random.default_rng(1000 * seed + d)
    U = U_ROWS
    if name == "a":
        I = 2000
        uf, vf = _grid(rng, (U, d), -4, 4, -3), _grid(rng, (I, d), -4, 4, -3)
        ub = _grid(rng, U, -16, 16, -6)
        z = _zero_rows(U)
        uf[z], ub[z] = 0.0, 0.0
        return _tables(3.0, ub, np.arange(I) * 2.0 ** -35, uf, vf), np.nonzero(z)[0]
    if name == "b":
        I = 2000
        return _tables(3.0, np.zeros(U), np.arange(I) * 2.0 ** -35, _grid(rng, (U, d), -4, 4, -25),
                       _grid(rng, (I, d), -4, 4, -3)), np.zeros(0, int)
    if name == "c":
        I = 2000
        return _tables(3.0, _grid(rng, U, -16, 16, -6), np.arange(I) * 2.0 ** -35, _grid(rng, (U, d), -4, 4, -3),
                       np.zeros((I, d))), np.arange(U)
    if name == "d":
        I = 2000
        # 1 + j * 2^-23 with j < 2^12: tf32 reads 1.0 whether it truncates or rounds to nearest (a j of 2^13 - 1 would
        # round up to 1 + 2^-10); the eight highest ids hold the largest j
        j = rng.integers(0, 2 ** 12 - 1, I)
        j[-8:] = 2 ** 12 - 1
        vf = np.repeat((1.0 + j * 2.0 ** -23)[:, None], d, axis=1)
        s = 2.0 ** -rng.integers(0, 5, U) * np.where(rng.random(U) < 0.8, 1.0, -1.0)
        return _tables(0.0, np.zeros(U), np.zeros(I), np.repeat(s[:, None], d, axis=1), vf), np.arange(U)
    if name == "e":
        I = 3000
        vf = 0.25 + _grid(rng, (I, d), -4, 4, -8).astype(np.float64)
        lo, hi = E_CLUSTER
        c = rng.integers(0, 32, hi - lo)              # within 2^-9 of each other, relative: inside E_u
        vf[lo:hi] = (1.0 + c * 2.0 ** -14)[:, None]
        s = 2.0 ** -rng.integers(0, 4, U) * np.where(rng.random(U) < 0.8, 1.0, -1.0)
        return _tables(0.0, np.zeros(U), np.zeros(I), np.repeat(s[:, None], d, axis=1), vf), np.nonzero(s > 0)[0]
    if name == "f":
        I = 2000
        return _tables(12000.0, _grid(rng, U, -256, 256, -6), 1000.0 + np.arange(I) * 0.25,
                       _grid(rng, (U, d), -8, 8, -4), _grid(rng, (I, d), -8, 8, -4)), np.zeros(0, int)
    raise ValueError(name)


FAMILIES = ["a", "b", "c", "d", "e", "f"]
# (family, k, n_cand): n_cand = k keeps no spare candidate; 128 is the largest buffer (AP_MAX_CAND)
CASES = [("a", 10, 24), ("b", 10, 24), ("c", 10, 24), ("d", 10, 24), ("e", 1, 1), ("e", 10, 10), ("e", 50, 128),
         ("f", 50, 64), ("f", 1, 1), ("f", 5, 8)]
EXCL_CASES = [("a", 10, 24), ("d", 10, 24), ("e", 10, 32), ("e", 1, 4)]


def exact_scores(t):
    """The float64 score matrix of als3.py:112, checked to be exact: a second summation order gives the same bits."""
    U64, V64 = t["user_feat"].astype(np.float64), t["item_feat"].astype(np.float64)
    ub, ib, mu = t["user_bias"].astype(np.float64), t["item_bias"].astype(np.float64), float(t["mu"][0])
    M = ((U64 @ V64.T + ub[:, None]) + ib[None, :]) + mu
    M2 = (V64[:, ::-1] @ U64[:, ::-1].T).T + (ub[:, None] + (ib[None, :] + mu))
    assert np.array_equal(M, M2), "inputs not exact in float64"
    return M


def ref_rank(M, k, excluded=None):
    """Ranking of each row (score descending, lowest id on ties) over its items not in excluded[u]; (-inf, -1) past them."""
    U, I = M.shape
    idx, val = np.full((U, k), -1, np.int32), np.full((U, k), -np.inf)
    for u in range(U):
        cand = np.arange(I)
        if excluded is not None and excluded[u]:
            keep = np.ones(I, bool)
            keep[list(excluded[u])] = False
            cand = cand[keep]
        order = cand[np.lexsort((cand, -M[u, cand]))][:k]
        idx[u, :len(order)], val[u, :len(order)] = order, M[u, order]
    return idx, val


def exclusion(M, k, n_cand, seed=0):
    """Every row's true top 3 (duplicated pairs for some rows), and row 1 keeps only m items, k < m < n_cand (when there
    is such an m).  -> (users, items, per-row sets, the short row or None)"""
    U, I = M.shape
    rng = np.random.default_rng(seed)
    top3 = ref_rank(M, 3)[0]
    users, items = np.repeat(np.arange(U), 3), top3.reshape(-1)
    users, items = np.concatenate([users, users[:30]]), np.concatenate([items, items[:30]])   # duplicated pairs
    short = None
    if n_cand - k >= 2:
        short, m = 1, (k + n_cand) // 2
        drop = rng.permutation(I)[m:]
        keep = users != short
        users, items = np.concatenate([users[keep], np.full(len(drop), short)]), np.concatenate([items[keep], drop])
    sets = [set() for _ in range(U)]
    for u, i in zip(users, items):
        sets[u].add(int(i))
    if short is not None:
        assert k < I - len(sets[short]) < n_cand
    return users.astype(np.int32), items.astype(np.int32), sets, short


# ---- the certificate's bound -------------------------------------------------------------------------------------------
def _vmax_bmax(t):
    V = np.sqrt((t["item_feat"].astype(np.float64) ** 2).sum(axis=1)).max()
    B = np.abs(t["item_bias"] + t["mu"][0]).max()           # float32 addition: fl(b_i + mu), as the sweep adds them
    return V, float(B)


def cert_bound(t):
    """E_u of allpairs_rescore_kernel, per user: (2^-9 + dim 2^-22) ||u|| V + 2^-22 (||u|| V + |b_u| + B), V = max ||v||,
    B = max |fl(b_i + mu)|."""
    d = t["user_feat"].shape[1]
    V, B = _vmax_bmax(t)
    uv = np.sqrt((t["user_feat"].astype(np.float64) ** 2).sum(axis=1)) * V
    return (2.0 ** -9 + d * 2.0 ** -22) * uv + 2.0 ** -22 * (uv + np.abs(t["user_bias"].astype(np.float64)) + B)


def old_bound(t):
    """The bound the certificate used before it covered the accumulation and the bias roundings: 2^-9 ||u|| V."""
    V, _ = _vmax_bmax(t)
    return 2.0 ** -9 * np.sqrt((t["user_feat"].astype(np.float64) ** 2).sum(axis=1)) * V


def _tf32(x, rounding):
    """fp32 -> tf32 (10 explicit mantissa bits): the low 13 bits truncated, or rounded to nearest even"""
    b = np.ascontiguousarray(x, np.float32).view(np.uint32)
    if rounding == "nearest":
        b = b + np.uint32(0xFFF) + ((b >> np.uint32(13)) & np.uint32(1))
    return (b & np.uint32(0xFFFFE000)).view(np.float32)


def model_tc_scores(t, rounding):
    """The sweep's score as a model: tf32 operands, exact products, the fp32 accumulator rounded after each 8-wide k-step,
    then fl(fl(acc + b_u) + fl(b_i + mu))."""
    Ut = _tf32(t["user_feat"], rounding).astype(np.float64)
    Vt = _tf32(t["item_feat"], rounding).astype(np.float64)
    acc = np.zeros((Ut.shape[0], Vt.shape[0]), np.float32)
    for k0 in range(0, Ut.shape[1], 8):
        acc = (acc + Ut[:, k0:k0 + 8] @ Vt[:, k0:k0 + 8].T).astype(np.float32)
    return (acc + t["user_bias"][:, None]) + (t["item_bias"] + t["mu"][0])[None, :]


@pytest.mark.parametrize("rounding", ["truncate", "nearest"])
@pytest.mark.parametrize("d", DIMS)
@pytest.mark.parametrize("fam", FAMILIES)
def test_bound_covers_the_modelled_tensor_core_score(fam, d, rounding):
    t, _ = family(fam, d)
    err = np.abs(model_tc_scores(t, rounding).astype(np.float64) - exact_scores(t))
    E = cert_bound(t)
    assert (err <= E[:, None]).all(), "worst excess %.3g" % (err - E[:, None]).max()


@pytest.mark.parametrize("fam", ["a", "b", "c"])
def test_tf32_only_bound_misses_the_bias_roundings(fam):
    """What the fix is for: on (a) - (c) the fp32 bias additions alone take the score further than 2^-9 ||u|| V."""
    t, _ = family(fam, 64)
    err = np.abs(model_tc_scores(t, "truncate").astype(np.float64) - exact_scores(t))
    assert (err > old_bound(t)[:, None]).any()


def test_exclusion_builder():
    t, _ = family("a", 32)
    M = exact_scores(t)
    users, items, sets, short = exclusion(M, 10, 24)
    assert short == 1 and 10 < M.shape[1] - len(sets[1]) < 24
    top3 = ref_rank(M, 3)[0]
    assert all(set(top3[u].tolist()) <= sets[u] for u in range(M.shape[0]) if u != 1)
    assert all(len(sets[u]) == 3 for u in range(M.shape[0]) if u != 1)


# ---- GPU --------------------------------------------------------------------------------------------------------------
def _engine(t):
    from tf_recomm_b200.engine import SvdEngine
    U, d = t["user_feat"].shape
    return SvdEngine(U, t["item_feat"].shape[0], d, 1e-3, 0.05, tables=t)


@pytest.mark.gpu
@pytest.mark.parametrize("d", DIMS)
@pytest.mark.parametrize("fam", FAMILIES)
def test_tensor_core_scores_stay_inside_the_bound(fam, d):
    """The premise of the certificate on the hardware: every tcgen05 kind::tf32 score is within E_u of the exact one."""
    t, _ = family(fam, d)
    s = _engine(t).allpairs(want_scores=True, want_best=False, use_tensor_cores=True)["scores"].cpu().numpy()
    err = np.abs(s.astype(np.float64) - exact_scores(t))
    E = cert_bound(t)
    assert (err <= E[:, None]).all(), "worst err / E %.4f" % (err / np.maximum(E[:, None], 1e-300)).max()


def _same_bits(a_idx, a_val, b_idx, b_val):
    assert np.array_equal(a_idx.cpu().numpy(), b_idx.cpu().numpy())
    assert np.array_equal(a_val.cpu().numpy().view(np.int64), b_val.cpu().numpy().view(np.int64))


def _assert_ranking(idx, val, ref_idx, ref_val, n_unc):
    got = idx.cpu().numpy()
    bad = np.nonzero((got != ref_idx).any(axis=1))[0]
    assert bad.size == 0, "%d rows differ, first %s (n_uncertified %d): got %s, float64 ranking %s" % (
        bad.size, bad[:8].tolist(), n_unc, got[bad[0]].tolist(), ref_idx[bad[0]].tolist())
    np.testing.assert_allclose(val.cpu().numpy(), ref_val, rtol=1e-12, atol=1e-12)


@pytest.mark.gpu
@pytest.mark.parametrize("d", DIMS)
@pytest.mark.parametrize("fam,k,n_cand", CASES)
def test_ranking_equals_float64_ranking(fam, k, n_cand, d):
    """rank_all_users = the float64 ranking, and rank_users returns its rows bit for bit; rows whose whole band of
    near-ties lies inside E_u go through the exact fallback."""
    t, forced = family(fam, d)
    M = exact_scores(t)
    ref_idx, ref_val = ref_rank(M, k)
    eng = _engine(t)
    idx, val, n_unc = eng.rank_all_users(k=k, n_cand=n_cand)
    _assert_ranking(idx, val, ref_idx, ref_val, n_unc)
    assert len(forced) <= n_unc <= M.shape[0]
    _same_bits(*eng.rank_users(np.arange(M.shape[0]), k=k), idx, val)
    # the exclusion entry with nothing excluded: the same bits
    _same_bits(*eng._rank_excluding(k, n_cand, None)[:2], idx, val)


@pytest.mark.gpu
@pytest.mark.parametrize("d", DIMS)
@pytest.mark.parametrize("fam,k,n_cand", EXCL_CASES)
def test_ranking_with_the_true_top_items_excluded(fam, k, n_cand, d):
    t, forced = family(fam, d)
    M = exact_scores(t)
    users, items, sets, short = exclusion(M, k, n_cand)
    ref_idx, ref_val = ref_rank(M, k, sets)
    eng = _engine(t)
    csr = eng.pair_csr(users, items)
    idx, val, n_unc = eng.rank_all_users(k=k, n_cand=n_cand, exclude=csr)
    _assert_ranking(idx, val, ref_idx, ref_val, n_unc)
    assert len(set(forced.tolist()) - {short}) <= n_unc
    _same_bits(*eng.rank_users(np.arange(M.shape[0]), k=k, exclude=csr), idx, val)


@pytest.mark.gpu
@pytest.mark.parametrize("d", [32, 128])
def test_ranking_metrics_against_the_true_top_k(d):
    """Family (a) with the held-out items = every user's float64 top-k: hit rate and precision are exactly 1."""
    k, n_cand = 10, 24
    t, forced = family("a", d)
    ref_idx, _ = ref_rank(exact_scores(t), k)
    U = ref_idx.shape[0]
    got = _engine(t).ranking_metrics(k, np.repeat(np.arange(U), k), ref_idx.reshape(-1), n_cand=n_cand)
    assert got["n_users"] == U
    assert got["hr"] == 1.0 and got["precision"] == 1.0 and got["recall"] == 1.0
    assert got["ndcg"] == pytest.approx(1.0, abs=1e-12)
    assert got["n_uncertified"] >= len(forced)


@pytest.mark.gpu
@pytest.mark.parametrize("d", [15, 160])
def test_exact_only_dims(d):
    """dims the tensor cores cannot take: every row through the exact float64 path, on family (a) and (g)."""
    k, n_cand = 10, 24
    t, _ = family("a", d)
    M = exact_scores(t)
    users, items, sets, _ = exclusion(M, k, n_cand)
    eng = _engine(t)
    for excl, ex in ((None, None), (sets, eng.pair_csr(users, items))):
        ref_idx, ref_val = ref_rank(M, k, excl)
        idx, val, n_unc = eng._rank_excluding(k, n_cand, ex)
        _assert_ranking(idx, val, ref_idx, ref_val, n_unc)
        assert n_unc == M.shape[0]
        _same_bits(*eng.rank_users(np.arange(M.shape[0]), k=k, exclude=ex), idx, val)
