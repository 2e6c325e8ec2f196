"""Implicit-feedback ALS on the device (iALS, Hu, Koren and Volinsky 2008): tfr_gram_rows / tfr_ials_half_sweep /
tfr_ials_objective (csrc/ials.cu), SvdEngine.ials_data / ials_sweep / implicit_objective / fold_in_implicit above them, and
svd_train_val.py --solver ials.  The numpy float64 reference below is one np.linalg.solve per row; it is pinned to the
gradient of the dense loss, with the confidence and preference matrices materialised over all U x I pairs."""
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
LAM = 0.05


# ---- numpy float64 reference -------------------------------------------------------------------------------------------------
def merge(rows, cols, w=None):
    """Distinct (row, col) pairs, weights summed (1 per entry by default) -> (rows, cols, w float64)."""
    w = np.ones(len(rows)) if w is None else np.asarray(w, np.float64)
    key, inv = np.unique(np.asarray(rows, np.int64) * (1 << 32) + np.asarray(cols, np.int64), return_inverse=True)
    ws = np.zeros(len(key))
    np.add.at(ws, inv, w)
    return key >> 32, key & 0xFFFFFFFF, ws


def half_ref(F, rows, cols, w, n_rows, alpha, lam):
    """Every row r in [0, n_rows) solved with the fixed side F: (F^T F + sum alpha w f f^T + lam I) x = sum (1 + alpha w) f
    over the merged pairs (rows == r).  -> [n_rows, d] float64, zeros for a row without interactions."""
    F = np.asarray(F, np.float64)
    d = F.shape[1]
    G = F.T @ F
    out = np.zeros((n_rows, d))
    for r in range(n_rows):
        sel = rows == r
        if not sel.any():
            continue
        Fs, ws = F[cols[sel]], w[sel]
        A = G + (Fs * (alpha * ws)[:, None]).T @ Fs + lam * np.eye(d)
        out[r] = np.linalg.solve(A, ((1.0 + alpha * ws)[:, None] * Fs).sum(0))
    return out


def dense(X, Y, users, items, w, alpha):
    """(C, P) over all U x I pairs from the merged interactions."""
    C, P = np.ones((len(X), len(Y))), np.zeros((len(X), len(Y)))
    C[users, items] = 1.0 + alpha * w
    P[users, items] = 1.0
    return C, P


def dense_loss(X, Y, users, items, w, alpha, lam):
    X, Y = np.asarray(X, np.float64), np.asarray(Y, np.float64)
    C, P = dense(X, Y, users, items, w, alpha)
    return float((C * (P - X @ Y.T) ** 2).sum() + lam * ((X ** 2).sum() + (Y ** 2).sum()))


def gram_loss(X, Y, users, items, w, alpha, lam):
    """The objective without the U x I matrix: sum (X^T X o Y^T Y) + sum_R [c (1 - s)^2 - s^2] + lam (tr + tr)."""
    X, Y = np.asarray(X, np.float64), np.asarray(Y, np.float64)
    Gx, Gy = X.T @ X, Y.T @ Y
    s = np.einsum("nd,nd->n", X[users], Y[items])
    return float((Gx * Gy).sum() + ((1.0 + alpha * w) * (1.0 - s) ** 2 - s ** 2).sum() + lam * (np.trace(Gx) + np.trace(Gy)))


# ---- CPU -------------------------------------------------------------------------------------------------------------------
def test_reference_half_steps_zero_the_dense_gradient():
    """U = 11, I = 9, d = 5 with duplicate pairs, the last user and item without interactions: after each reference
    half-step, the gradient of the dense loss vanishes for that side's rows; a perturbed row's does not; the Gram-trick
    objective equals the dense one."""
    rng = np.random.default_rng(0)
    U, I, d, alpha, lam = 11, 9, 5, 4.0, 0.3
    n = 40
    users, items = rng.integers(0, U - 1, n), rng.integers(0, I - 1, n)
    users[:4], items[:4] = users[4], items[4]
    mu, mi, mw = merge(users, items, rng.integers(1, 5, n) / 4.0)
    assert len(mu) < n
    X, Y = rng.normal(0, 0.3, (U, d)), rng.normal(0, 0.3, (I, d))

    def grad(X, Y):
        C, P = dense(X, Y, mu, mi, mw, alpha)
        R = C * (P - X @ Y.T)
        return -2 * R @ Y + 2 * lam * X, -2 * R.T @ X + 2 * lam * Y, np.abs(2 * (C * P) @ Y).max() + 1.0
    L = dense_loss(X, Y, mu, mi, mw, alpha, lam)
    assert abs(gram_loss(X, Y, mu, mi, mw, alpha, lam) - L) <= 1e-12 * L
    X = half_ref(Y, mu, mi, mw, U, alpha, lam)
    gx, _, scale = grad(X, Y)
    assert np.abs(gx).max() <= 1e-10 * scale
    assert not X[U - 1].any()
    Y = half_ref(X, mi, mu, mw, I, alpha, lam)
    _, gy, scale = grad(X, Y)
    assert np.abs(gy).max() <= 1e-10 * scale
    assert not Y[I - 1].any()
    L = dense_loss(X, Y, mu, mi, mw, alpha, lam)
    assert abs(gram_loss(X, Y, mu, mi, mw, alpha, lam) - L) <= 1e-12 * L
    Y[2] += 0.1   # a perturbed row: the test has teeth
    _, gy, scale = grad(X, Y)
    assert np.abs(gy[2]).max() > 1e-3 * scale


def _half(L, dim=16, reg=0.05, alpha=1.0, n_light=3, n_heavy=1, n_chunks=2, feat=1, fixed=1, gram=1, failed=1, ws=1,
          ws_bytes=1 << 30, chunk=64, weight=1, stride=0):
    """tfr_ials_half_sweep with dummy (never dereferenced) pointers: only the argument checks can run."""
    p = 4096
    return L.tfr_ials_half_sweep(fixed and p, 100, dim, stride, gram and p, alpha, reg, p, p, weight and p, p, n_light, p, p,
                                 n_heavy, p, n_chunks, chunk, feat and p, 0, None, failed and p, ws and p, ws_bytes, None)


def test_invalid_arguments_are_refused_before_any_cuda_call():
    L = _lib.load()
    bad = (dict(dim=0), dict(dim=129), dict(reg=0.0), dict(reg=-1.0), dict(reg=float("nan")), dict(reg=float("inf")),
           dict(alpha=-1.0), dict(alpha=float("nan")), dict(alpha=float("inf")), dict(feat=0), dict(fixed=0), dict(gram=0),
           dict(failed=0), dict(weight=0), dict(ws=0), dict(chunk=0), dict(n_chunks=0), dict(stride=8))
    for kw in bad:
        assert _half(L, **kw) == -1, kw   # TFR_ERR_INVALID
    assert _half(L, ws_bytes=100) == -3   # TFR_ERR_WORKSPACE, still before any CUDA call
    assert _half(L, n_light=0, n_heavy=0, n_chunks=0, feat=0, fixed=0, gram=0, failed=0, ws=0, weight=0) == 0   # a no-op
    p = 4096

    def gram(dim=16, n=100, feat=p, out=p, ws=p, nbytes=1 << 30, stride=0):
        return L.tfr_gram_rows(feat, n, dim, stride, out, ws, nbytes, None)
    for kw in (dict(dim=0), dict(dim=129), dict(n=-1), dict(feat=0), dict(out=0), dict(ws=0), dict(stride=8)):
        assert gram(**kw) == -1, kw
    assert gram(nbytes=100) == -3

    def obj(dim=16, reg=0.05, alpha=1.0, out=p, ws=p, nbytes=1 << 30, ug=p, ig=p, w=p):
        return L.tfr_ials_objective(p, p, 10, 10, dim, 0, 0, ug, ig, alpha, reg, p, p, w, out, ws, nbytes, None)
    for kw in (dict(dim=0), dict(dim=129), dict(reg=0.0), dict(reg=float("nan")), dict(alpha=-1.0),
               dict(alpha=float("inf")), dict(out=0), dict(ws=0), dict(ug=0), dict(ig=0), dict(w=0)):
        assert obj(**kw) == -1, kw
    assert obj(nbytes=10) == -3


def test_workspace_sizes():
    L = _lib.load()
    assert L.tfr_ials_workspace_bytes(1, 128) >= (128 * 129 // 2 + 128) * 8 == 67072
    assert L.tfr_ials_workspace_bytes(1000, 128) >= 1000 * 67072
    assert L.tfr_ials_workspace_bytes(-1, 8) < 0 and L.tfr_ials_workspace_bytes(1, 129) < 0
    assert L.tfr_gram_workspace_bytes(0, 128) >= 0
    assert L.tfr_gram_workspace_bytes(4097, 128) >= 5 * 128 * 129 // 2 * 8   # one partial per 1024 rows
    assert L.tfr_gram_workspace_bytes(-1, 8) < 0 and L.tfr_gram_workspace_bytes(10, 0) < 0
    assert L.tfr_ials_objective_workspace_bytes(10 ** 6) >= 1024 * 2 * 8 and L.tfr_ials_objective_workspace_bytes(-1) < 0


@pytest.mark.skipif(not os.path.exists(NVCC), reason="needs the CUDA toolkit")
def test_ials_kernels_compile_without_spills(tmp_path):
    from test_rank_users import _ptxas_lines
    info = {}
    for src in ("ials.cu", "als.cu"):   # als.cu: the half-sweep kernels, one template with ALS's
        obj, log = str(tmp_path / (src + ".o")), str(tmp_path / (src + ".txt"))
        with open(log, "w") as f:
            subprocess.check_call([NVCC, "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-ccbin",
                                   "/usr/bin/g++", "-Xcompiler", "-fPIC", "-Xptxas", "-v", "-c",
                                   os.path.join(ROOT, "tf-recomm_b200", "csrc", src), "-o", obj],
                                  stdout=f, stderr=subprocess.STDOUT)
        info.update(_ptxas_lines(log))
    half_sweep = ["void tfr::half_sweep_%s_kernel<tfr::FiForm<false, true, false> >" % k   # FiImplicit
                  for k in ("rows", "chunk_gram", "heavy_solve")]
    names = {"tfr::gram_rows_kernel", "tfr::gram_combine_kernel", *half_sweep, "tfr::ials_objective_rows_kernel",
             "tfr::ials_objective_finish_kernel"}
    assert names <= set(info), sorted(info)
    for name in names:
        assert tuple(info[name][1:]) == (0, 0, 0), (name, info[name])
    for name in ("tfr::gram_rows_kernel", *half_sweep):
        assert info[name][0] <= 128, (name, info[name])   # __launch_bounds__(256, 2): two CTAs per SM


@pytest.mark.parametrize("extra", [["--variant", "fork", "--topk", "10"], []])
def test_driver_refuses_before_device_work(extra, capsys):
    import svd_train_val
    with pytest.raises(SystemExit):
        svd_train_val.main(["--synthetic", "ml1m", "--solver", "ials", "--epochs", "1"] + extra)
    assert "--solver ials" in capsys.readouterr().err


# ---- GPU -------------------------------------------------------------------------------------------------------------------
def _gram_call(eng_L, feat2d, n, d, stride):
    import torch
    out = torch.empty(d * (d + 1) // 2, dtype=torch.float64, device=feat2d.device)
    nbytes = _lib.check(eng_L.tfr_gram_workspace_bytes(n, d))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=feat2d.device)
    _lib.check(eng_L.tfr_gram_rows(feat2d.data_ptr(), n, d, stride, out.data_ptr(), ws.data_ptr(), nbytes,
                                   torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return out.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("d", [1, 15, 32, 100, 128])
def test_gram_rows_against_numpy(d):
    """Every entry within 1e-12 of sum |x_a x_b| of numpy's float64 Gram, on a strided table, and the same bits twice."""
    import torch
    L = _lib.load()
    rng = np.random.default_rng(d)
    stride = d + 3
    for n in (0, 1, 4095, 4097, 162541):
        F = rng.normal(0, 0.5, (n, stride)).astype(np.float32)
        Fd = torch.from_numpy(F).cuda()
        got = _gram_call(L, Fd, n, d, stride)
        X = F[:, :d].astype(np.float64)
        ref, bound = X.T @ X, np.abs(X).T @ np.abs(X)
        ia, ib = np.tril_indices(d)
        order = np.lexsort((ib, ia))   # packed row-major lower triangle
        ia, ib = ia[order], ib[order]
        assert (np.abs(got - ref[ia, ib]) <= 1e-12 * bound[ia, ib]).all(), (n, d)
        assert np.array_equal(got.view(np.uint64), _gram_call(L, Fd, n, d, stride).view(np.uint64)), (n, d)


def _interactions(U, I, d, seed, heavy):
    """Users 0..5 with 0, 1, d - 1, d, d + 1 and `heavy` interactions, items 0..5 the same from filler users (>= 8), fillers
    among themselves; a duplicate in every row of two or more, and weights in quarters (exact sums)."""
    rng = np.random.default_rng(seed)
    us, its = [], []
    for k, c in enumerate([0, 1, max(d - 1, 0), d, d + 1, heavy]):
        f = rng.integers(8, I, c)
        if c >= 2:
            f[-1] = f[0]
        us.append(np.full(c, k)); its.append(f)
        g = rng.integers(8, U, c)
        if c >= 2:
            g[-1] = g[0]
        us.append(g); its.append(np.full(c, k))
    us.append(rng.integers(8, U, 4000)); its.append(rng.integers(8, I, 4000))
    users, items = np.concatenate(us).astype(np.int32), np.concatenate(its).astype(np.int32)
    perm = rng.permutation(len(users))
    return users[perm], items[perm], (rng.integers(1, 9, len(users)) / 4.0).astype(np.float32)


def _engine(U, I, d, seed=5, reg=LAM, **kw):
    from tf_recomm_b200 import init
    from tf_recomm_b200.engine import SvdEngine
    tabs = init.init_tables(U, I, d, seed=seed, bias_init="truncated_normal")
    tabs["user_feat"] *= 10
    tabs["item_feat"] *= 10
    tabs["mu"][:] = 3.5
    return SvdEngine(U, I, d, 1e-3, reg, tables=tabs, **kw)


def _tables(eng):
    return {n: eng.t[n].cpu().numpy().copy() for n in ("mu", "user_bias", "item_bias", "user_feat", "item_feat")}


def _user_half(eng, data, alpha, reg=LAM):
    import torch
    T = eng.t
    with torch.cuda.device(eng.device):
        eng._gram(T["item_feat"], eng.I, data.item_gram, data.workspace)
        eng._ials_half(data, alpha, reg, data.by_user, data.user_plan, (T["item_feat"], eng.I, data.item_gram),
                       (T["user_feat"], T["user_bias"]))


def _item_half(eng, data, alpha, reg=LAM):
    import torch
    T = eng.t
    with torch.cuda.device(eng.device):
        eng._gram(T["user_feat"], eng.U, data.user_gram, data.workspace)
        eng._ials_half(data, alpha, reg, data.by_item, data.item_plan, (T["user_feat"], eng.U, data.user_gram),
                       (T["item_feat"], T["item_bias"]))


def _check_rows(got, ref):
    """test_als._check_rows's bar: 2^-24 |ref| + 1e-10 max |ref| per entry."""
    got = got.astype(np.float64)
    for r in range(len(ref)):
        tol = 2.0 ** -24 * np.abs(ref[r]) + 1e-10 * np.abs(ref[r]).max()
        assert (np.abs(got[r] - ref[r]) <= tol).all(), (r, np.abs(got[r] - ref[r]).max(), np.abs(ref[r]).max())


class _Chunk:
    def __init__(self, v):
        self.v = v

    def __enter__(self):
        self.old = _lib.tune_get("ALS_CHUNK")
        _lib.tune_set("ALS_CHUNK", self.v)

    def __exit__(self, *a):
        _lib.tune_set("ALS_CHUNK", self.old)


@pytest.mark.gpu
@pytest.mark.parametrize("d", [1, 8, 15, 64, 128])
@pytest.mark.parametrize("alpha", [0.0, 1.0, 40.0])
def test_half_steps_match_numpy(d, alpha):
    """Each half-step against np.linalg.solve from the GPU's own tables just before it, within 2^-24 |ref| + 1e-10 max|ref|,
    for rows with 0, 1, d - 1, d, d + 1 and more than ALS_CHUNK (64) interactions; the fixed side is unchanged bit for bit,
    solved rows' biases are exactly 0, and a whole sweep leaves mu = 0."""
    U, I = 300, 200
    users, items, w = _interactions(U, I, d, seed=d, heavy=300)
    mu_, mi_, mw_ = merge(users, items, w)
    lam = float(np.float32(LAM))
    with _Chunk(64):
        eng = _engine(U, I, d)
        data = eng.ials_data(users, items, w)
    assert data.chunk == 64 and data.user_plan.heavy.numel() >= 1 and data.item_plan.heavy.numel() >= 1
    assert data.by_user.partner.numel() == len(mu_)
    T0 = _tables(eng)
    _user_half(eng, data, alpha)
    T1 = _tables(eng)
    _check_rows(T1["user_feat"], half_ref(T0["item_feat"], mu_, mi_, mw_, U, alpha, lam))
    assert not T1["user_bias"].any() and not T1["user_feat"][0].any()
    assert all(np.array_equal(T0[n], T1[n]) for n in ("mu", "item_feat", "item_bias"))
    _item_half(eng, data, alpha)
    T2 = _tables(eng)
    _check_rows(T2["item_feat"], half_ref(T1["user_feat"], mi_, mu_, mw_, I, alpha, lam))
    assert not T2["item_bias"].any() and not T2["item_feat"][0].any()
    assert all(np.array_equal(T1[n], T2[n]) for n in ("mu", "user_feat", "user_bias"))
    assert int(data.failed.item()) == 0
    assert int(eng.ials_sweep(data, alpha).item()) == 0
    assert _tables(eng)["mu"][0] == 0.0


@pytest.mark.gpu
def test_chunked_and_one_cta_paths_agree_and_keep_their_bits():
    """The same rows solved through the chunked path (ALS_CHUNK = 32) and the one-CTA path agree within the bar; the chunked
    result is the same bits run to run and in a CUDA-graph replay of ials_sweep."""
    import torch
    U, I, d, alpha = 300, 200, 32, 10.0
    users, items, w = _interactions(U, I, d, seed=11, heavy=500)
    eng = _engine(U, I, d)
    start = _tables(eng)

    def restore(e):
        for n, a in start.items():
            e.t[n].copy_(torch.from_numpy(a.reshape(e.t[n].shape)))
    with _Chunk(1 << 20):
        big = eng.ials_data(users, items, w)
    with _Chunk(32):
        small = eng.ials_data(users, items, w)
    assert big.user_plan.heavy.numel() == 0 and small.user_plan.heavy.numel() >= 1
    _user_half(eng, big, alpha)
    one = eng.t["user_feat"].cpu().numpy().copy()
    restore(eng)
    _user_half(eng, small, alpha)
    split = eng.t["user_feat"].cpu().numpy().copy()
    mu_, mi_, mw_ = merge(users, items, w)
    ref = half_ref(start["item_feat"], mu_, mi_, mw_, U, alpha, float(np.float32(LAM)))
    _check_rows(one, ref)
    _check_rows(split, ref)
    restore(eng)
    _user_half(eng, small, alpha)
    assert np.array_equal(split.view(np.uint32), eng.t["user_feat"].cpu().numpy().view(np.uint32))

    def sweep_bits():
        torch.cuda.synchronize()
        return [v.view(np.uint8) for v in _tables(eng).values()]
    restore(eng)
    eng.ials_sweep(small, alpha)
    first = sweep_bits()
    restore(eng)
    eng.ials_sweep(small, alpha)
    assert all(np.array_equal(a, b) for a, b in zip(first, sweep_bits()))
    restore(eng)
    exe = eng._capture(lambda: eng.ials_sweep(small, alpha))
    try:
        restore(eng)
        _lib.check(eng.L.tfr_graph_launch(exe, torch.cuda.current_stream(eng.device).cuda_stream))
        assert all(np.array_equal(a, b) for a, b in zip(first, sweep_bits()))
    finally:
        eng.L.tfr_graph_destroy(exe)


@pytest.mark.gpu
@pytest.mark.parametrize("sgd", [False, True])
def test_fold_in_implicit_equals_the_user_half_sweep(sgd):
    """Training users folded in from their own interactions (duplicates unmerged: fold_in_implicit merges them the same way)
    get the user half-sweep's bits, so rank_folded ranks them as rank_users does."""
    import torch
    U, I, d, alpha = 300, 200, 64, 5.0
    users, items, w = _interactions(U, I, d, seed=3, heavy=100)
    eng = _engine(U, I, d, flags=_lib.OPT_SGD if sgd else 0)
    data = eng.ials_data(users, items, w)
    assert data.user_plan.heavy.numel() == 0
    eng.ials_sweep(data, alpha)   # a trained model: both sides solved
    f = eng.fold_in_implicit(users, items, w, n=U, alpha=alpha)
    _user_half(eng, data, alpha)
    assert np.array_equal(f.feat.cpu().numpy().view(np.uint32), eng.t["user_feat"].cpu().numpy().view(np.uint32))
    assert not f.bias.cpu().numpy().any() and not f.info.cpu().numpy().any()
    q = torch.arange(U, dtype=torch.int32, device=eng.device)
    ia, va = eng.rank_folded(f, k=20)
    ib, vb = eng.rank_users(q, k=20, exclude=(users, items))
    assert np.array_equal(ia.cpu().numpy(), ib.cpu().numpy())
    assert np.array_equal(va.cpu().numpy(), vb.cpu().numpy())


@pytest.mark.gpu
def test_objective_matches_numpy_and_never_rises():
    """The objective against numpy's (rel <= 1e-12), then over 5 sweeps the loss after each half-step is <= the loss before
    it times (1 + 1e-7): each half-step is an exact block minimisation in float64, and rounding the solved rows to fp32
    moves the loss by a second-order amount far below that tolerance."""
    U, I, d, alpha = 400, 300, 16, 10.0
    rng = np.random.default_rng(1)
    users, items = rng.integers(0, U, 20000).astype(np.int32), rng.integers(0, I, 20000).astype(np.int32)
    eng = _engine(U, I, d)
    eng.t["user_feat"].mul_(5)
    data = eng.ials_data(users, items)
    mu_, mi_, mw_ = merge(users, items)
    lam = float(np.float32(LAM))

    def check_np():
        o = eng.implicit_objective(data, alpha)
        T = _tables(eng)
        want = gram_loss(T["user_feat"], T["item_feat"], mu_, mi_, mw_, alpha, lam)
        assert abs(o["loss"] - want) <= 1e-12 * want, (o, want)
        assert abs(o["loss"] - dense_loss(T["user_feat"], T["item_feat"], mu_, mi_, mw_, alpha, lam)) <= 1e-12 * want
        assert o["n"] == len(mu_)
        assert abs(o["loss"] - (o["all_pairs"] + o["observed"] + o["penalty"])) <= 1e-15 * o["loss"]
        return o["loss"]
    prev = first = check_np()
    for _ in range(5):
        for step in (_user_half, _item_half):
            step(eng, data, alpha)
            cur = eng.implicit_objective(data, alpha)["loss"]
            assert cur <= prev * (1 + 1e-7), (step.__name__, prev, cur)
            prev = cur
    assert prev < first
    check_np()


@pytest.mark.gpu
def test_planted_clusters_are_recovered():
    """Disjoint user / item clusters, every user interacting with every item of its cluster but one, held out: after 3
    sweeps, ranking_metrics(k = 10, exclude = train) puts the held-out item in the top 10 for >= 95% of users."""
    rng = np.random.default_rng(7)
    n_clusters, upc, ipc, d = 8, 40, 30, 16
    U, I = n_clusters * upc, n_clusters * ipc
    tu, ti, vu, vi = [], [], [], []
    for u in range(U):
        c = u // upc
        its = c * ipc + rng.permutation(ipc)
        tu += [u] * (ipc - 1); ti += list(its[1:]); vu.append(u); vi.append(its[0])
    eng = _engine(U, I, d)
    data = eng.ials_data(tu, ti)
    for _ in range(3):
        assert int(eng.ials_sweep(data, 10.0, reg=0.1).item()) == 0
    m = eng.ranking_metrics(10, vu, vi, exclude=(tu, ti))
    assert m["n_users"] == U and m["hr"] >= 0.95, m


@pytest.mark.gpu
def test_unsupported_models_and_arguments_are_refused():
    from tf_recomm_b200.engine import SvdEngine, TfrError
    users, items = np.array([0, 1]), np.array([1, 0])
    for kw in (dict(flags=_lib.ABS_ITEM), dict(flags=_lib.LOSS_SIGMOID_CE), dict(var_mask=_lib.VAR_UF | _lib.VAR_IF),
               dict(d=129)):
        d = kw.pop("d", 8)
        eng = SvdEngine(4, 4, d, 1e-3, 0.05, **kw)
        with pytest.raises(TfrError):
            eng.ials_data(users, items)
    eng = SvdEngine(4, 4, 8, 1e-3, 0.05)
    for w in ([1.0, 0.0], [1.0, -1.0], [1.0, float("nan")], [1.0, float("inf")]):
        with pytest.raises(TfrError):
            eng.ials_data(users, items, w)
    data = eng.ials_data(users, items)
    for alpha, reg in ((1.0, 0.0), (1.0, float("nan")), (-1.0, 0.1), (float("inf"), 0.1)):
        with pytest.raises(TfrError):
            eng.ials_sweep(data, alpha, reg=reg)
    with pytest.raises(TfrError):
        eng.ials_data([0, 4], [1, 0])


@pytest.mark.gpu
def test_driver_ials(tmp_path):
    import svd_train_val
    from tf_recomm_b200.engine import SvdEngine
    ckpt = str(tmp_path / "ials.ckpt")
    buf = io.StringIO()
    with redirect_stdout(buf):
        svd_train_val.main(["--synthetic", "ml1m", "--ratings", "100000", "--solver", "ials", "--alpha", "10", "--epochs",
                            "4", "--dim", "15", "--checkpoint", ckpt, "--logdir", str(tmp_path / "log"), "--topk", "10"])
    out = buf.getvalue()
    loss = [float(m) for m in re.findall(r"IMPLICIT\(pairs=\d+, loss=([-0-9.e+]+)", out)]
    assert len(loss) == 4 and all(np.isfinite(loss)), out
    assert all(b <= a * (1 + 1e-7) for a, b in zip(loss, loss[1:])), loss
    assert out.count("TOPK(k=10") == 4
    assert os.listdir(str(tmp_path / "log"))
    eng = SvdEngine.from_checkpoint(ckpt)
    assert eng.d == 15 and not eng.t["user_bias"].cpu().numpy().any() and eng.t["mu"].item() == 0.0
