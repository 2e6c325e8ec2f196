"""Fold-in of users the model was not trained on: tfr_fold_in_users (csrc/fold_in.cu), SvdEngine.fold_in / rank_folded above
it, and recommend.py --fold-in.  The objective is the training loss restricted to one user with the item side fixed; the numpy
reference below is pinned to the training step's own gradients (oracle/np_oracle.py::grads)."""
import ctypes as C
import io
import os
import subprocess
import sys
from contextlib import redirect_stdout

import numpy as np
import pytest

from oracle import np_oracle
from tf_recomm_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NVCC = "/usr/local/cuda/bin/nvcc"
FLAG_SETS = [0, _lib.ABS_ITEM, _lib.REG_BIAS, _lib.ABS_ITEM | _lib.REG_BIAS]


# ---- numpy float64 reference -------------------------------------------------------------------------------------------------
def fold_system(V, ib, mu, items, rates, reg, flags):
    """The fold-in normal equations of one user in float64: (A, b) with A = sum_j x_j x_j^T + reg * n * D,
    b = sum_j (r_j - mu - b_{i_j}) x_j, x_j = [v~_{i_j} ; 1]."""
    d = V.shape[1]
    X = V[items].astype(np.float64)
    if flags & _lib.ABS_ITEM:
        X = np.abs(X)
    X = np.hstack([X, np.ones((len(items), 1))])
    Dg = np.ones(d + 1)
    Dg[d] = 1.0 if flags & _lib.REG_BIAS else 0.0
    A = X.T @ X + float(np.float32(reg)) * len(items) * np.diag(Dg)
    y = (rates.astype(np.float64) - float(mu)) - ib[items].astype(np.float64)
    return A, X.T @ y


def fold_ref(V, ib, mu, items, rates, reg, flags):
    """-> theta = [p_u ; b_u] in float64 (zeros for a row without ratings)."""
    if len(items) == 0:
        return np.zeros(V.shape[1] + 1)
    A, b = fold_system(V, ib, mu, items, rates, reg, flags)
    return np.linalg.solve(A, b)


# ---- CPU -------------------------------------------------------------------------------------------------------------------
def _call(L, dim=16, flags=0, reg=0.05, n=3, feat=1, bias=1, info=1, indptr=1):
    """tfr_fold_in_users with dummy (never dereferenced) pointers: only the argument checks can run."""
    p = 4096
    return L.tfr_fold_in_users(p, p, p, 100, dim, 0, flags, reg, indptr and p, p, p, n, feat and p, bias and p,
                               info and p, None)


def test_invalid_arguments_are_refused_before_any_cuda_call():
    L = _lib.load()
    for kw in (dict(dim=0), dict(dim=129), dict(flags=_lib.LOSS_SIGMOID_CE), dict(flags=_lib.FORK_FLAGS), dict(reg=-1.0),
               dict(reg=float("nan")), dict(reg=float("inf")), dict(feat=0), dict(bias=0), dict(info=0), dict(indptr=0)):
        assert _call(L, **kw) == -1, kw   # TFR_ERR_INVALID
    assert _call(L, n=0, feat=0, bias=0, info=0, indptr=0) == 0   # n = 0: a no-op


@pytest.mark.parametrize("flags", FLAG_SETS)
def test_reference_solution_zeroes_the_training_gradients(flags):
    """The reference's theta makes the oracle's per-occurrence user gradients, summed over the user's ratings (duplicates
    included), vanish: the fold-in objective is the training objective."""
    rng = np.random.default_rng(flags)
    I, d, reg = 60, 15, np.float32(0.05)
    p = dict(mu=np.array([3.5], np.float32), user_bias=np.zeros(1, np.float32),
             item_bias=rng.normal(0, 0.5, I).astype(np.float32), user_feat=np.zeros((1, d), np.float32),
             item_feat=rng.normal(0, 0.3, (I, d)).astype(np.float32))
    n = 29
    items = rng.integers(0, I, n)
    items[:4] = items[4]
    rates = rng.integers(1, 6, n).astype(np.float32)
    th = fold_ref(p["item_feat"], p["item_bias"], p["mu"][0], items, rates, reg, flags)
    p["user_feat"][0], p["user_bias"][0] = th[:d], th[d]
    g = np_oracle.grads(p, np.zeros(n, np.int64), items, rates, reg, abs_item=bool(flags & _lib.ABS_ITEM),
                        reg_bias=bool(flags & _lib.REG_BIAS))
    _, b = fold_system(p["item_feat"], p["item_bias"], p["mu"][0], items, rates, reg, flags)
    scale = np.abs(b).max()
    assert np.abs(g["g_uf"].astype(np.float64).sum(0)).max() < 1e-5 * scale
    assert abs(float(g["g_ub"].astype(np.float64).sum())) < 1e-5 * scale
    # and a different row does not: the test has teeth
    p["user_bias"][0] += 0.1
    g = np_oracle.grads(p, np.zeros(n, np.int64), items, rates, reg, abs_item=bool(flags & _lib.ABS_ITEM),
                        reg_bias=bool(flags & _lib.REG_BIAS))
    assert abs(float(g["g_ub"].astype(np.float64).sum())) > 1e-2


@pytest.mark.skipif(not os.path.exists(NVCC), reason="needs the CUDA toolkit")
def test_fold_in_kernel_compiles_without_spills(tmp_path):
    from test_rank_users import _ptxas_lines
    obj, log = str(tmp_path / "fold_in.o"), str(tmp_path / "ptxas.txt")
    with open(log, "w") as f:
        subprocess.check_call([NVCC, "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-ccbin",
                               "/usr/bin/g++", "-Xcompiler", "-fPIC", "-Xptxas", "-v", "-c",
                               os.path.join(ROOT, "tf-recomm_b200", "csrc", "fold_in.cu"), "-o", obj],
                              stdout=f, stderr=subprocess.STDOUT)
    info = _ptxas_lines(log)
    assert "tfr::fold_in_kernel" in info, sorted(info)
    regs, stack, st, ld = info["tfr::fold_in_kernel"]
    assert (stack, st, ld) == (0, 0, 0), info
    assert regs <= 128, regs   # __launch_bounds__(256, 2): two CTAs per SM


# ---- GPU -------------------------------------------------------------------------------------------------------------------
def _engine(U, I, d, flags=0, seed=31, reg=0.05):
    from tf_recomm_b200 import init
    from tf_recomm_b200.engine import SvdEngine
    tabs = init.init_tables(U, I, d, seed=seed, bias_init="truncated_normal")
    tabs["item_feat"] *= 25
    tabs["user_feat"] *= 25
    tabs["item_bias"] *= 10
    tabs["mu"][:] = 3.5
    return SvdEngine(U, I, d, 1e-3, reg, flags=flags, tables=tabs), tabs


def _rows(I, d, counts, seed=0):
    """Rating rows of the given sizes, duplicates in every row of two or more, shuffled across rows.
    -> (rows, items, rates) as host arrays."""
    rng = np.random.default_rng(seed)
    rows, items = [], []
    for r, c in enumerate(counts):
        it = rng.integers(0, I, c)
        if c >= 2:
            it[-1] = it[0]
        rows.append(np.full(c, r))
        items.append(it)
    rows, items = np.concatenate(rows), np.concatenate(items)
    rates = rng.integers(1, 6, len(rows)).astype(np.float32)
    perm = rng.permutation(len(rows))
    return rows[perm], items[perm].astype(np.int32), rates[perm]


def _bits(*arrays):
    return [np.ascontiguousarray(a.cpu().numpy()).view(np.uint8).copy() for a in arrays]


@pytest.mark.gpu
@pytest.mark.parametrize("d", [1, 15, 20, 32, 128])
@pytest.mark.parametrize("flags", FLAG_SETS)
@pytest.mark.parametrize("reg", [0.05, 1e-3])
def test_fold_in_matches_numpy(d, flags, reg):
    """Every output entry within 2^-24 |ref| + 1e-10 max|ref| of np.linalg.solve on the same float64 system, for rows
    with 1, 2, d, d + 1, d + 2 and several thousand ratings."""
    I = 3000
    eng, tabs = _engine(40, I, d, flags=flags, reg=reg)
    counts = [1, 2, d, d + 1, d + 2, 3001, 5, 70]
    rows, items, rates = _rows(I, d, counts, seed=d + flags)
    f = eng.fold_in(rows, items, rates)
    assert (f.info.cpu().numpy() == 0).all()
    feat, bias = f.feat.cpu().numpy(), f.bias.cpu().numpy()
    for r in range(len(counts)):
        sel = rows == r
        ref = fold_ref(tabs["item_feat"], tabs["item_bias"], tabs["mu"][0], items[sel], rates[sel], reg, flags)
        got = np.append(feat[r].astype(np.float64), float(bias[r]))
        tol = 2.0 ** -24 * np.abs(ref) + 1e-10 * np.abs(ref).max()
        assert (np.abs(got - ref) <= tol).all(), (r, counts[r], np.abs(got - ref).max(), np.abs(ref).max())


@pytest.mark.gpu
def test_a_rows_bits_do_not_depend_on_the_batch():
    """A row folded alone, inside a batch of 4096 and inside a permuted batch gives the same bits; two calls agree."""
    I, d = 5000, 128
    eng, _ = _engine(10, I, d)
    rng = np.random.default_rng(3)
    counts = rng.integers(0, 400, 4096)
    counts[17] = 2500
    rows, items, rates = _rows(I, d, counts, seed=4)
    full = eng.fold_in(rows, items, rates)
    again = eng.fold_in(rows, items, rates)
    assert all(np.array_equal(a, b) for a, b in zip(_bits(full.feat, full.bias, full.info),
                                                     _bits(again.feat, again.bias, again.info)))
    inv = np.argsort(rng.permutation(4096))             # row r of the batch becomes row inv[r]
    pf = eng.fold_in(inv[rows], items, rates, n=4096)
    want = _bits(full.feat, full.bias)
    got = _bits(pf.feat[inv], pf.bias[inv])
    assert all(np.array_equal(a, b) for a, b in zip(want, got))
    for r in (17, 0, 4095):
        sel = rows == r
        one = eng.fold_in(np.zeros(sel.sum(), np.int64), items[sel], rates[sel])
        assert np.array_equal(_bits(one.feat)[0], _bits(full.feat[r:r + 1])[0])
        assert np.array_equal(_bits(one.bias)[0], _bits(full.bias[r:r + 1])[0])


def _c_fold(eng, indptr, items, rates, reg, flags=None, stream=None, out=None):
    """tfr_fold_in_users straight from the C ABI on device CSR arrays -> (feat, bias, info)."""
    import torch
    n = indptr.numel() - 1
    if out is None:
        out = (torch.empty(n, eng.d, device=eng.device), torch.empty(n, device=eng.device),
               torch.empty(n, dtype=torch.int32, device=eng.device))
    st = stream if stream is not None else torch.cuda.current_stream(eng.device).cuda_stream
    T = eng.t
    _lib.check(eng.L.tfr_fold_in_users(T["item_feat"].data_ptr(), T["item_bias"].data_ptr(), T["mu"].data_ptr(), eng.I,
                                       eng.d, eng.feat_stride, eng.flags if flags is None else flags, reg,
                                       indptr.data_ptr(), items.data_ptr(), rates.data_ptr(), n, out[0].data_ptr(),
                                       out[1].data_ptr(), out[2].data_ptr(), st))
    return out


@pytest.mark.gpu
def test_edge_rows():
    import torch
    from tf_recomm_b200.engine import TfrError
    I, d = 400, 20
    eng, tabs = _engine(10, I, d)
    dev = eng.device
    # an empty row (row 1 of 3): zeros, info 0
    f = eng.fold_in(np.array([0, 2, 2]), np.array([5, 6, 7]), np.array([4.0, 3.0, 1.0], np.float32), n=3)
    assert (f.feat[1] == 0).all() and float(f.bias[1]) == 0.0 and (f.info.cpu().numpy() == 0).all()
    assert eng.fold_in([], [], []).feat.shape == (0, d)
    # host-side checks
    with pytest.raises(TfrError):
        eng.fold_in([0, 1], [3, I], [1.0, 2.0])
    with pytest.raises(TfrError):
        eng.fold_in([0, 3], [3, 4], [1.0, 2.0], n=3)
    with pytest.raises(TfrError):
        eng.fold_in([0, 1], [3, 4], [1.0])
    # C level: an out-of-range id in row 1 gives info -1 and a NaN row; rows 0 and 2 are unchanged
    indptr = torch.tensor([0, 3, 6, 9], dtype=torch.int64, device=dev)
    items = torch.tensor([1, 2, 3, 4, I, 5, 6, 7, 8], dtype=torch.int32, device=dev)
    rates = torch.tensor([5, 4, 3, 2, 1, 2, 3, 4, 5], dtype=torch.float32, device=dev)
    feat, bias, info = _c_fold(eng, indptr, items, rates, 0.05)
    assert info.cpu().tolist() == [0, -1, 0]
    assert torch.isnan(feat[1]).all() and torch.isnan(bias[1])
    ok = eng.fold_in(np.repeat([0, 1], 3), np.array([1, 2, 3, 6, 7, 8]), np.array([5, 4, 3, 3, 4, 5], np.float32))
    assert torch.equal(feat[[0, 2]], ok.feat) and torch.equal(bias[[0, 2]], ok.bias)
    # reg = 0 with the row's item vectors zeroed: the first pivot is exactly 0.0.  Row 1 is unregularised too, so it needs
    # d + 1 independent ratings or more to be solvable (one rating alone gives a rank-one matrix: pivot 2 fails)
    eng2, tabs2 = _engine(10, I, d)
    eng2.t["item_feat"][[10, 11]] = 0
    it1 = np.arange(100, 100 + 3 * (d + 1))
    r1 = np.random.default_rng(8).integers(1, 6, len(it1)).astype(np.float32)
    z = eng2.fold_in(np.r_[0, 0, np.ones(len(it1), np.int64)], np.r_[10, 11, it1], np.r_[np.float32([3, 4]), r1],
                     reg=0.0)
    assert z.info.cpu().tolist() == [1, 0]
    assert torch.isnan(z.feat[0]).all() and torch.isnan(z.bias[0]) and not torch.isnan(z.feat[1]).any()
    ref = fold_ref(tabs2["item_feat"], tabs2["item_bias"], tabs2["mu"][0], it1, r1, 0.0, 0)
    np.testing.assert_allclose(np.append(z.feat[1].cpu().numpy(), z.bias[1].cpu().numpy()), ref, rtol=1e-5, atol=1e-6)
    one = eng2.fold_in([0], [12], [5.0], reg=0.0)   # rank one: the first pivot is > 0, the second is not
    assert one.info.cpu().tolist() == [2] and torch.isnan(one.feat).all()
    idx, val = eng2.rank_folded(z, k=5)
    assert (idx[0] == -1).all() and torch.isneginf(val[0]).all() and (idx[1] >= 0).all()
    # the fork's loss is refused
    fork, _ = _engine(10, I, d, flags=_lib.FORK_FLAGS)
    with pytest.raises(TfrError):
        fork.fold_in([0], [1], [1.0])


@pytest.mark.gpu
@pytest.mark.parametrize("flags", [0, _lib.ABS_ITEM])
def test_rank_folded_equals_rank_users_of_the_written_rows(flags):
    """rank_folded = rank_users(ids, exclude=the folded pairs) once the folded rows are written into the user table at ids,
    in item ids and float64 bits; ABS_ITEM scores by u.|v|."""
    from test_rank_users import _same
    U, I, d, k = 300, 2500, 64, 30
    eng, _ = _engine(U, I, d, flags=flags)
    counts = [0, 1, 5, 64, 80, 700, 2400, 12]   # row 6 has nearly every item rated
    rows, items, rates = _rows(I, d, counts, seed=9)
    f = eng.fold_in(rows, items, rates)
    ids = np.array([250, 3, 77, 12, 299, 0, 140, 41])
    eng.t["user_feat"][ids] = f.feat
    eng.t["user_bias"][ids] = f.bias
    for excl in (True, False):
        want = eng.rank_users(ids, k=k, exclude=(ids[rows], items) if excl else None)
        _same(eng.rank_folded(f, k=k, exclude_rated=excl), want)
    got_i = eng.rank_folded(f, k=k)[0].cpu().numpy()
    for r in range(len(counts)):
        assert not set(got_i[r].tolist()) & set(items[rows == r].tolist())


@pytest.mark.gpu
def test_graph_capture_and_replay_with_new_ratings():
    import torch
    I, d = 2000, 32
    eng, _ = _engine(10, I, d)
    rows, items, rates = _rows(I, d, [40, 1, 300, 33], seed=11)
    f = eng.fold_in(rows, items, rates)
    indptr, it_d = f.ratings.indptr, f.ratings.items.clone()
    rt_d = torch.empty(len(rates), dtype=torch.float32, device=eng.device)
    rng = np.random.default_rng(12)
    cap = torch.cuda.Stream(device=eng.device)
    cap.wait_stream(torch.cuda.current_stream(eng.device))
    exe = C.c_void_p()
    with torch.cuda.stream(cap):
        _lib.check(eng.L.tfr_graph_begin_capture(cap.cuda_stream))
        try:
            g_out = _c_fold(eng, indptr, it_d, rt_d, 0.05, stream=cap.cuda_stream)
        finally:
            rc = eng.L.tfr_graph_end_capture(cap.cuda_stream, C.byref(exe))
        _lib.check(rc)
    torch.cuda.current_stream(eng.device).wait_stream(cap)
    try:
        for _ in range(2):
            it_d.copy_(torch.from_numpy(rng.integers(0, I, it_d.numel()).astype(np.int32)))
            rt_d.copy_(torch.from_numpy(rng.integers(1, 6, rt_d.numel()).astype(np.float32)))
            _lib.check(eng.L.tfr_graph_launch(exe, torch.cuda.current_stream(eng.device).cuda_stream))
            eager = _c_fold(eng, indptr, it_d, rt_d, 0.05)
            torch.cuda.synchronize(eng.device)
            assert all(np.array_equal(a, b) for a, b in zip(_bits(*g_out), _bits(*eager)))
    finally:
        eng.L.tfr_graph_destroy(exe)


def _train_checkpoint(tmp_path, ratings, epochs, dim=20):
    import svd_train_val
    ckpt = str(tmp_path / "model.ckpt")
    data = ["--synthetic", "ml1m", "--ratings", str(ratings)]
    with redirect_stdout(io.StringIO()):
        svd_train_val.main(data + ["--epochs", str(epochs), "--dim", str(dim), "--checkpoint", ckpt, "--logdir",
                                   str(tmp_path / "log")])
    return ckpt, data


def _train_split(ratings):
    from tf_recomm_b200 import config, synthetic
    U, I, _ = synthetic.SHAPES["ml1m"]
    au, ai, ar = synthetic.make_ratings(U, I, ratings, seed=config.SEED)
    (tu, ti, tr), _ = synthetic.split(au, ai, ar)
    return tu, ti, tr


@pytest.mark.gpu
def test_fold_in_minimises_the_training_loss(tmp_path):
    """Trained for a few epochs at the ML-1M shape, every user folded in from their own training ratings: the float64 user
    part of the training loss at the folded row is no larger than at the trained row, and its gradient vanishes up to the
    fp32 rounding of the row."""
    from tf_recomm_b200 import config
    from tf_recomm_b200.engine import SvdEngine
    ckpt, _ = _train_checkpoint(tmp_path, 100000, 3)
    eng = SvdEngine.from_checkpoint(ckpt)
    tu, ti, tr = _train_split(100000)
    reg = config.LAMBDA_REG
    f = eng.fold_in(tu, ti, tr, n=eng.U, reg=reg)
    assert (f.info.cpu().numpy() == 0).all()
    T = {n: eng.t[n].cpu().numpy().astype(np.float64) for n in ("mu", "user_bias", "item_bias", "user_feat", "item_feat")}
    feat, bias = f.feat.cpu().numpy().astype(np.float64), f.bias.cpu().numpy().astype(np.float64)
    regd = float(np.float32(reg))
    order = np.argsort(tu, kind="stable")
    starts = np.searchsorted(tu[order], np.arange(eng.U + 1))
    checked = 0
    for u in range(eng.U):
        sel = order[starts[u]:starts[u + 1]]
        if len(sel) == 0:
            assert not feat[u].any() and bias[u] == 0.0
            continue
        V = T["item_feat"][ti[sel]]
        y = (tr[sel].astype(np.float64) - T["mu"][0]) - T["item_bias"][ti[sel]]

        def loss(p, b):
            e = V @ p + b - y
            return 0.5 * (e @ e) + 0.5 * regd * len(sel) * (p @ p)

        assert loss(feat[u], bias[u]) <= loss(T["user_feat"][u], T["user_bias"][u]) * (1 + 1e-9), u
        A, rhs = fold_system(T["item_feat"], T["item_bias"], T["mu"][0], ti[sel], tr[sel], reg, 0)
        th = np.append(feat[u], bias[u])
        grad = A @ th - rhs
        bound = 2.0 ** -22 * (np.abs(A) @ np.abs(th) + np.abs(rhs))
        assert (np.abs(grad) <= bound).all(), (u, np.abs(grad).max(), bound.min())
        checked += 1
    assert checked > 5000


# ---- recommend.py ------------------------------------------------------------------------------------------------------------
def _parse(text):
    out = []
    for line in text.splitlines():
        u, _, rest = line.partition("\t")
        pairs = [p.split(":") for p in rest.split()]
        out.append((u, [int(i) for i, _ in pairs], [float(v) for _, v in pairs]))
    return out


@pytest.mark.gpu
def test_recommend_cli_fold_in(tmp_path):
    import recommend
    from tf_recomm_b200 import config
    from tf_recomm_b200.engine import SvdEngine
    ckpt, data = _train_checkpoint(tmp_path, 20000, 1)
    tu, ti, tr = _train_split(20000)
    eng = SvdEngine.from_checkpoint(ckpt)
    u7 = tu == 7
    rng = np.random.default_rng(2)
    csv = tmp_path / "new.csv"
    lines = ["user,item,rating"]
    lines += ["bob,%d,%g" % (i, r) for i, r in zip(rng.integers(0, eng.I, 6), rng.integers(1, 6, 6))]
    lines += ["user 7,%d,%g" % (i, r) for i, r in zip(ti[u7], tr[u7])]
    lines += ["bob,12,5", "42,100,3"]
    csv.write_text("\n".join(lines) + "\n")
    run = subprocess.run([sys.executable, os.path.join(ROOT, "recommend.py"), "--checkpoint", ckpt, "--fold-in", str(csv),
                          "--k", "10"], capture_output=True, text=True, cwd=ROOT)
    assert run.returncode == 0, run.stderr
    out = _parse(run.stdout)
    assert [u for u, _, _ in out] == ["bob", "user 7", "42"]
    assert all(len(items) == 10 for _, items, _ in out)
    # the training user's ratings under a new label: exactly rank_folded of their fold-in
    f = eng.fold_in(np.zeros(u7.sum(), np.int64), ti[u7], tr[u7], reg=config.LAMBDA_REG)
    idx, val = (x.cpu().numpy()[0] for x in eng.rank_folded(f, k=10))
    assert out[1][1] == idx.tolist()
    np.testing.assert_allclose(out[1][2], val, rtol=0, atol=5.1e-7)
    assert not set(out[1][1]) & set(ti[u7].tolist())
    assert 12 not in out[0][1] and 100 not in out[2][1]
    buf = io.StringIO()
    recommend.main(["--checkpoint", ckpt, "--fold-in", str(csv), "--k", "10", "--no-exclude"], out=buf)
    f = eng.fold_in(np.zeros(u7.sum(), np.int64), ti[u7], tr[u7], reg=config.LAMBDA_REG)
    idx = eng.rank_folded(f, k=10, exclude_rated=False)[0].cpu().numpy()[0]
    assert _parse(buf.getvalue())[1][1] == idx.tolist()
    # --users is unchanged: the rank_users ranking with the training split excluded
    buf = io.StringIO()
    recommend.main(["--checkpoint", ckpt, "--users", "3,7", "--k", "10"] + data, out=buf)
    idx, val = (x.cpu().numpy() for x in eng.rank_users([3, 7], k=10, exclude=(tu, ti)))
    for r, (u, items, scores) in enumerate(_parse(buf.getvalue())):
        assert u == str([3, 7][r]) and items == idx[r][idx[r] >= 0].tolist()
        np.testing.assert_allclose(scores, val[r][idx[r] >= 0], rtol=0, atol=5.1e-7)
    # exactly one of --users / --fold-in
    for argv in (["--checkpoint", ckpt], ["--checkpoint", ckpt, "--users", "3", "--fold-in", str(csv)]):
        with pytest.raises(SystemExit):
            recommend.main(argv, out=io.StringIO())
