"""Ranking of unseen items and top-k recommendation metrics: tfr_allpairs_rank_excluding (each user's excluded items never
ranked, any dim <= 512), tfr_ranking_metrics (hit rate / precision / recall / NDCG at k on the device), the engine calls
above them (SvdEngine.rank_all_users(exclude=...), ranking_metrics) and the driver's --topk report."""
import io
import os
import re
import subprocess
from contextlib import redirect_stdout

import numpy as np
import pytest

from tf_recomm_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NVCC = "/usr/local/cuda/bin/nvcc"
CUOBJDUMP = "/usr/local/cuda/bin/cuobjdump"


# ---- numpy references ---------------------------------------------------------------------------------------------------
def ref_metrics(topk_idx, relevant):
    """(sum HR, sum precision, sum recall, sum NDCG, rows evaluated) and the per-row [n, 4] values (NaN where the row has
    no relevant item) of a ranking topk_idx [n, k] (-1 = no item) against relevant[u] = set of item ids."""
    n, k = topk_idx.shape
    rows = np.full((n, 4), np.nan)
    sums = np.zeros(5)
    disc = 1.0 / np.log2(np.arange(k) + 2.0)
    for u in range(n):
        rel = relevant[u]
        if not rel:
            continue
        h = np.array([x >= 0 and int(x) in rel for x in topk_idx[u]], dtype=np.float64)
        hits = h.sum()
        rows[u] = (float(hits >= 1), hits / k, hits / len(rel), (h * disc).sum() / disc[:min(k, len(rel))].sum())
        sums[:4] += rows[u]
        sums[4] += 1
    return sums, rows


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
def test_ranking_metrics_workspace_query_needs_no_gpu():
    L = _lib.load()
    assert L.tfr_ranking_metrics_workspace_bytes(162541, 50) > 0
    assert L.tfr_ranking_metrics_workspace_bytes(0, 50) > 0
    assert L.tfr_ranking_metrics_workspace_bytes(-1, 50) < 0
    assert L.tfr_ranking_metrics_workspace_bytes(10, 0) < 0


def test_reference_metrics_hand_worked_example():
    """k = 3.  User 0 ranks [5, 2, 7] with relevant {2, 9}: one hit at rank 1.  User 1 ranks [4, -1, -1] (one rankable
    item) with relevant {4}: a hit at rank 0, and the ideal list has one entry.  User 2 has no relevant item: not
    evaluated."""
    topk = np.array([[5, 2, 7], [4, -1, -1], [0, 1, 2]], np.int32)
    sums, rows = ref_metrics(topk, [{2, 9}, {4}, set()])
    d1 = 1.0 / np.log2(3.0)                                # discount of rank 1
    ndcg0 = d1 / (1.0 + d1)
    np.testing.assert_allclose(rows[0], [1.0, 1.0 / 3, 0.5, ndcg0], rtol=1e-15)
    np.testing.assert_allclose(rows[1], [1.0, 1.0 / 3, 1.0, 1.0], rtol=1e-15)
    assert np.isnan(rows[2]).all()
    np.testing.assert_allclose(sums, [2.0, 2.0 / 3, 1.5, 1.0 + ndcg0, 2.0], rtol=1e-15)
    assert abs(ndcg0 - 0.38685280723454163) < 1e-15


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


@pytest.mark.skipif(not (os.path.exists(NVCC) and os.path.exists(CUOBJDUMP)), reason="needs the CUDA toolkit")
def test_exclusion_sweep_compiles_to_tcgen05_without_spills(tmp_path):
    """The EXCL instantiations of allpairs_tc_kernel are still the tcgen05 sweep (UTCHMMA, LDTM, UTMALDG in the SASS) and
    spill nothing; the existing instantiations keep their register counts (94 / 108 / 150 / 158 with CUDA 12.9)."""
    obj = str(tmp_path / "allpairs.o")
    log = str(tmp_path / "ptxas.txt")
    with open(log, "w") as f:
        subprocess.check_call([NVCC, "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-ccbin",
                               "/usr/bin/g++", "-Xcompiler", "-fPIC", "-Xptxas", "-v", "-c",
                               os.path.join(ROOT, "tf-recomm_b200", "csrc", "allpairs.cu"), "-o", obj],
                              stdout=f, stderr=subprocess.STDOUT)
    info = _ptxas_lines(log)
    tc = {k: v for k, v in info.items() if "allpairs_tc_kernel<" in k}
    assert len(tc) == 20, sorted(tc)
    existing = {(False, False): 94, (False, True): 108, (True, False): 150, (True, True): 158}
    for kc in (1, 2, 3, 4):
        for (topk, obs), regs in existing.items():
            name = "void tfr::allpairs_tc_kernel<%d, %s, %s, false>" % (kc, str(topk).lower(), str(obs).lower())
            if "release 12.9" in subprocess.run([NVCC, "--version"], capture_output=True, text=True).stdout:
                assert tc[name][0] == regs, (name, tc[name])
            assert tc[name][2:] == [0, 0], (name, tc[name])
        excl = tc["void tfr::allpairs_tc_kernel<%d, true, false, true>" % kc]
        assert excl[2:] == [0, 0], excl
    sass = subprocess.run([CUOBJDUMP, "-sass", obj], capture_output=True, text=True, check=True).stdout
    blocks = re.split(r"\n\s*Function : ", sass)
    excl_blocks = [b for b in blocks if b.startswith("_ZN3tfr18allpairs_tc_kernelILi") and "ELb1ELb0ELb1E" in b.split()[0]]
    assert len(excl_blocks) == 4
    for b in excl_blocks:
        for op in ("UTCHMMA", "LDTM", "UTMALDG"):
            assert op in b, (b.split()[0], op)


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


def _zipf_ids(rng, n, size, a=1.0):
    p = 1.0 / np.arange(1, n + 1) ** a
    p /= p.sum()
    return rng.permutation(n)[rng.choice(n, size=size, p=p)].astype(np.int32)


def _exclusion_pairs(M, kk, seed=0):
    """Zipf-drawn pairs with duplicates + every user's unmasked top-3; user 0: every item; user 1: I - kk + 3 items (fewer
    than kk rankable: padded; I - 1 when kk <= 3); the last three users: nothing.  -> (users, items) shuffled, and the
    per-user sets."""
    U, I = M.shape
    n1 = min(I - kk + 3, I - 1)
    rng = np.random.default_rng(seed)
    n = 4 * U
    users, items = _zipf_ids(rng, U, n, 0.8), _zipf_ids(rng, I, n, 1.0)
    users, items = np.concatenate([users, users[:50]]), np.concatenate([items, items[:50]])   # duplicated pairs
    top3 = np.stack([np.lexsort((np.arange(I), -M[u]))[:3] for u in range(U)])
    users, items = np.concatenate([users, np.repeat(np.arange(U), 3)]), np.concatenate([items, top3.reshape(-1)])
    keep = (users != 1) & (users < U - 3)
    x1 = rng.choice(I, n1, replace=False)
    users = np.concatenate([users[keep], np.zeros(I, np.int64), np.ones(n1 + len(x1[:5]), np.int64)]).astype(np.int32)
    items = np.concatenate([items[keep], np.arange(I), x1, x1[:5]]).astype(np.int32)
    perm = rng.permutation(len(users))
    users, items = users[perm], items[perm]
    sets = [set() for _ in range(U)]
    for u, i in zip(users, items):
        sets[u].add(int(i))
    assert len(sets[0]) == I and len(sets[1]) == n1 and not sets[U - 1]
    return users, items, sets


def _check_masked(U, I, d, k, n_cand, ties):
    eng, tabs = _engine(U, I, d, ties)
    M = _f64_scores(tabs)
    kk = min(k, I)
    users, items, sets = _exclusion_pairs(M, kk)
    idx, val, n_unc = eng.rank_all_users(k=k, n_cand=n_cand, exclude=(users, items))
    ref_idx, ref_val = ref_rank_excluding(M, kk, sets)
    got = idx.cpu().numpy()
    assert got.shape == (U, kk)
    assert np.array_equal(got, ref_idx), "%d rows differ (n_uncertified %d)" % (int((got != ref_idx).any(axis=1).sum()), n_unc)
    np.testing.assert_allclose(val.cpu().numpy(), ref_val, rtol=1e-12, atol=1e-12)
    r1 = I - len(sets[1])                       # user 1's rankable items: kk - 3 when kk > 3
    assert (got[0] == -1).all() and (got[1, r1:] == -1).all() and (got[1, :min(r1, kk)] >= 0).all()
    return eng, n_unc


@pytest.mark.gpu
@pytest.mark.parametrize("U,I,d,k,n_cand,ties", [(300, 1000, 64, 50, 64, 0), (129, 777, 128, 50, 64, 5),
                                                 (257, 40, 32, 50, 64, 0), (64, 3000, 96, 1, 8, 5),
                                                 (500, 2048, 128, 10, 16, 0), (70, 900, 64, 50, 64, 1)])
def test_masked_ranking_equals_float64_ranking(U, I, d, k, n_cand, ties):
    """rank_all_users(exclude=...) = the float64 ranking of every user's remaining items (excluded entries removed, lowest
    id on ties), whatever tf32 did; ties = 1 sends every row that has k rankable ties through the exact fallback."""
    _, n_unc = _check_masked(U, I, d, k, n_cand, ties)
    if ties == 1:
        assert n_unc >= U - 2     # all but user 0 (nothing rankable) and user 1 (fewer than n_cand rankable: no drops)
    assert 0 <= n_unc <= U


@pytest.mark.gpu
@pytest.mark.parametrize("d", [15, 20, 48, 160])
def test_masked_ranking_at_dims_the_tensor_cores_cannot_take(d):
    """dim % 32 != 0 or dim > 128: every row goes through the exact float64 path, same result."""
    _, n_unc = _check_masked(150, 700, d, 20, 32, 0)
    assert n_unc == 150


@pytest.mark.gpu
@pytest.mark.parametrize("d", [64, 20])
def test_masked_ranking_of_the_fork_model_scores_abs_item_features(d):
    """The fork variant's model scores u.|v| + biases (ABS_ITEM): its unseen-item ranking is the float64 ranking of that."""
    eng, tabs = _engine(200, 600, d, flags=_lib.FORK_FLAGS)
    tabs = dict(tabs, item_feat=np.abs(tabs["item_feat"]))
    M = _f64_scores(tabs)
    users, items, sets = _exclusion_pairs(M, 20)
    idx, val, _ = eng.rank_all_users(k=20, n_cand=32, exclude=(users, items))
    ref_idx, ref_val = ref_rank_excluding(M, 20, sets)
    assert np.array_equal(idx.cpu().numpy(), ref_idx)
    np.testing.assert_allclose(val.cpu().numpy(), ref_val, rtol=1e-12, atol=1e-12)


@pytest.mark.gpu
@pytest.mark.parametrize("U,I,d,k,n_cand,ties", [(300, 1000, 64, 50, 64, 0), (70, 900, 64, 50, 64, 1),
                                                 (500, 2048, 128, 10, 16, 0)])
def test_rank_without_exclusion_is_bit_identical_through_both_entries(U, I, d, k, n_cand, ties):
    eng, _ = _engine(U, I, d, ties)
    a_idx, a_val, a_unc = eng.rank_all_users(k=k, n_cand=n_cand)                  # tfr_allpairs_consume
    b_idx, b_val, b_unc = eng._rank_excluding(k, n_cand, None)                      # tfr_allpairs_rank_excluding, null list
    assert np.array_equal(a_idx.cpu().numpy(), b_idx.cpu().numpy())
    assert np.array_equal(a_val.cpu().numpy().view(np.int64), b_val.cpu().numpy().view(np.int64))
    assert a_unc == b_unc


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_ranking_sums_match_numpy_and_repeat_bit_identically(seed):
    """tfr_ranking_metrics on random rankings (with -1 entries and duplicate-free rows) against the numpy reference."""
    import torch
    from tf_recomm_b200.engine import PairCSR
    rng = np.random.default_rng(seed)
    U, I, k = 3000 + seed, 500, [1, 10, 50][seed]
    eng, _ = _engine(U, I, 32)
    topk = np.stack([rng.permutation(I)[:k] for _ in range(U)]).astype(np.int32)
    topk[rng.random((U, k)) < 0.05] = -1
    n_rel = rng.integers(0, 30, U)
    n_rel[:5] = 0
    ru = np.repeat(np.arange(U), n_rel)
    ri = np.concatenate([rng.choice(I, n, replace=False) for n in n_rel]).astype(np.int32)
    rel = eng.pair_csr(ru, ri)
    rows = torch.empty(U, 4, dtype=torch.float64, device=eng.device)
    t = torch.from_numpy(topk).to(eng.device)
    s1 = eng.ranking_sums(t, rel, row_metrics=rows).cpu().numpy()
    s2 = eng.ranking_sums(t, PairCSR(rel.indptr, rel.items)).cpu().numpy()
    sets = [set() for _ in range(U)]
    for u, i in zip(ru, ri):
        sets[u].add(int(i))
    ref_s, ref_rows = ref_metrics(topk, sets)
    np.testing.assert_allclose(s1, ref_s, rtol=1e-12)
    np.testing.assert_allclose(rows.cpu().numpy(), ref_rows, rtol=1e-12)
    assert np.array_equal(s1.view(np.int64), s2.view(np.int64))


@pytest.mark.gpu
@pytest.mark.parametrize("U,I,d,k,min_rating", [(400, 1500, 64, 20, None), (300, 600, 20, 10, 4.0), (129, 777, 128, 50, 3.0)])
def test_ranking_metrics_match_numpy(U, I, d, k, min_rating):
    """ranking_metrics: rank with the training pairs excluded, score against the held-out pairs minus the excluded ones."""
    eng, tabs = _engine(U, I, d)
    M = _f64_scores(tabs)
    rng = np.random.default_rng(U)
    tu, ti = _zipf_ids(rng, U, 6 * U, 0.8), _zipf_ids(rng, I, 6 * U, 1.0)
    vu, vi = _zipf_ids(rng, U, 3 * U, 0.8), _zipf_ids(rng, I, 3 * U, 1.0)
    vu, vi = np.concatenate([vu, tu[:20], vu[:10]]), np.concatenate([vi, ti[:20], vi[:10]])   # overlap + duplicates
    vr = rng.integers(1, 6, len(vu)).astype(np.float32)
    got = eng.ranking_metrics(k, vu, vi, rates=vr, min_rating=min_rating, exclude=(tu, ti))
    excl = [set() for _ in range(U)]
    for u, i in zip(tu, ti):
        excl[u].add(int(i))
    rel = [set() for _ in range(U)]
    for u, i, r in zip(vu, vi, vr):
        if (min_rating is None or r >= min_rating) and int(i) not in excl[u]:
            rel[u].add(int(i))
    ref_idx, _ = ref_rank_excluding(M, min(k, I), excl)
    s, _ = ref_metrics(ref_idx, rel)
    assert got["n_users"] == int(s[4]) > 0
    for j, key in enumerate(("hr", "precision", "recall", "ndcg")):
        assert got[key] == pytest.approx(s[j] / s[4], rel=1e-12), key
    again = eng.ranking_metrics(k, vu, vi, rates=vr, min_rating=min_rating, exclude=eng.pair_csr(tu, ti))
    for key in ("hr", "precision", "recall", "ndcg", "n_users"):
        assert got[key] == again[key]


# ---- the driver's --topk report ------------------------------------------------------------------------------------------
def _run(argv):
    import svd_train_val
    buf = io.StringIO()
    with redirect_stdout(buf):
        svd_train_val.main(argv)
    return buf.getvalue()


def _report_lines(text):
    return [l for l in text.splitlines() if re.match(r"^\s*\d+ TRAIN\(", l)]


TOPK_RE = (r"^TOPK\(k=(\d+), users=(\d+), hr=([0-9.]+), precision=([0-9.]+), recall=([0-9.]+), ndcg=([0-9.]+)\)$")


@pytest.mark.gpu
@pytest.mark.parametrize("dim", [15, 32])
def test_driver_topk_report(tmp_path, dim):
    """--topk 10 in both modes: the RMSE report lines are those of the run without it (elapsed time aside), one TOPK line
    follows each, the evaluated users are those with a validation item rated >= 4 that they did not rate in training, and
    the last recall beats a random ranking of the same users' unseen items."""
    from tf_recomm_b200 import config, summary, synthetic
    K = 10
    common = ["--synthetic", "ml1m", "--ratings", "60000", "--epochs", "2", "--dim", str(dim)]
    U, I, _ = synthetic.SHAPES["ml1m"]
    users, items, rates = synthetic.make_ratings(U, I, 60000, seed=config.SEED)
    (tu, ti, _), (vu, vi, vr) = synthetic.split(users, items, rates)
    seen = set(zip(tu.tolist(), ti.tolist()))
    rel = {}
    for u, i, r in zip(vu.tolist(), vi.tolist(), vr.tolist()):
        if r >= 4.0 and (u, i) not in seen:
            rel.setdefault(u, set()).add(i)
    n_seen = np.bincount(np.unique(tu.astype(np.int64) * I + ti) // I, minlength=U)
    random_recall = np.mean([min(1.0, K / (I - n_seen[u])) for u in rel])
    strip = lambda l: re.sub(r" [0-9.]+\(s\)$", "", l)   # noqa: E731
    for mode in ("session", "stream"):
        tag = "%s%d" % (mode, dim)
        plain = _run(common + ["--mode", mode, "--checkpoint", os.devnull, "--logdir", ""])
        text = _run(common + ["--mode", mode, "--topk", str(K), "--checkpoint", os.devnull,
                              "--logdir", str(tmp_path / tag)])
        assert [strip(l) for l in _report_lines(plain)] == [strip(l) for l in _report_lines(text)]
        lines = text.splitlines()
        at = [j for j, l in enumerate(lines) if re.match(r"^\s*\d+ TRAIN\(", l)]
        assert len(at) >= 2
        tops = []
        for j in at:
            m = re.match(TOPK_RE, lines[j + 1])
            assert m, lines[j + 1]
            tops.append(m)
        assert all(int(m.group(1)) == K and int(m.group(2)) == len(rel) for m in tops)
        assert float(tops[-1].group(5)) > random_recall, (tops[-1].group(0), random_recall)
        ev = summary.read_events(str(next((tmp_path / tag).iterdir())))
        for name, g in (("hr_at_k", 3), ("precision_at_k", 4), ("recall_at_k", 5), ("ndcg_at_k", 6)):
            vals = [v for _, t, v in ev if t == name]
            assert len(vals) == len(tops)
            assert vals[-1] == pytest.approx(float(tops[-1].group(g)), abs=2e-6)


@pytest.mark.gpu
def test_driver_topk_report_fork_variant(tmp_path):
    """DISCRETE branch: an outcome of 1 in the validation split is relevant; the report follows each ACC / AUC line."""
    from tf_recomm_b200 import config, synthetic
    U, I, _ = synthetic.SHAPES["ml1m"]
    users, items, rates = synthetic.make_ratings(U, I, 30000, seed=config.SEED, binary=True)
    (tu, ti, _), (vu, vi, vr) = synthetic.split(users, items, rates)
    seen = set(zip(tu.tolist(), ti.tolist()))
    n_rel = len({u for u, i, r in zip(vu.tolist(), vi.tolist(), vr.tolist()) if r == 1.0 and (u, i) not in seen})
    text = _run(["--synthetic", "ml1m", "--ratings", "30000", "--epochs", "2", "--batch", "500", "--dim", "20",
                 "--variant", "fork", "--lr", "0.005", "--reg", "0.01", "--topk", "5", "--checkpoint", os.devnull,
                 "--logdir", ""])
    lines = text.splitlines()
    at = [j for j, l in enumerate(lines) if re.match(r"^\s*\d+ TRAIN\(size=\d+/\d+, macc=", l)]
    assert len(at) >= 2
    for j in at:
        m = re.match(TOPK_RE, lines[j + 1])
        assert m and int(m.group(1)) == 5 and int(m.group(2)) == n_rel, lines[j + 1]
