"""KTM encoder + FM train-step oracle (CPU) and the CUDA FM step against the oracle (GPU, through the C ABI).

Pinned by the reference: the encoder against the known-answer table typeset in diagram_pretty.tex:16-22,31
(tests/golden/ktm_encoder_dummy.json).  FM TRAINING parity is unpinned (the reference trains with libFM's MCMC,
fm.py:154-155: external binary, random, no golden vectors): the oracle's FM step is checked against torch-CPU
autograd, the CUDA step against the oracle."""
import json
import os

import numpy as np
import pytest
import scipy.sparse as sp
import torch

import oracle
from tf_recomm_b200 import _lib, dataio, ktm

RTOL = 1e-5


# ---- CPU: encoder ----------------------------------------------------------------------------------------------------
def _dummy(golden_dir):
    import pandas as pd
    g = json.load(open(os.path.join(golden_dir, "ktm_encoder_dummy.json")))
    rows = np.array(g["rows_user_item_outcome"])
    df = pd.DataFrame(dict(user=rows[:, 0], item=rows[:, 1], outcome=rows[:, 2].astype(np.float32),
                           wins=0, fails=0))
    return g, df, sp.csr_matrix(np.array(g["qmatrix"]))


def test_encoder_reproduces_diagram_pretty_tex(golden_dir):
    g, df, q = _dummy(golden_dir)
    sw, sf = ktm.skill_counters(df["user"], df["item"], df["outcome"], q)
    X = ktm.df_to_sparse(df, g["blocks"], 2, 3, q, sw, sf)
    assert X.shape == (7, sum(g["block_widths"]))
    assert np.array_equal(X.toarray(), np.array(g["X"], dtype=np.float64))
    assert list(df["outcome"].astype(int)) == g["outcome"]


def test_encoder_blocks_follow_active_agents_order(golden_dir):
    g, df, q = _dummy(golden_dir)
    sw, sf = ktm.skill_counters(df["user"], df["item"], df["outcome"], q)
    full = np.array(g["X"], dtype=np.float64)
    X = ktm.df_to_sparse(df, ["users", "items"], 2, 3, q)           # IRT / MIRTb encoding: two-hot rows
    assert np.array_equal(X.toarray(), full[:, :5]) and (X.getnnz(axis=1) == 2).all()
    X = ktm.df_to_sparse(df, ["skills", "attempts"], 2, 3, q, sw, sf)  # AFM
    assert np.array_equal(X.toarray(), np.hstack([full[:, 5:8], full[:, 8:11] + full[:, 11:14]]))
    X = ktm.df_to_sparse(df, ["items"], 2, 3, None)                 # no q-matrix -> identity (fm.py:45-46)
    assert np.array_equal(X.toarray(), full[:, 2:5])
    with pytest.raises(ValueError):
        ktm.df_to_sparse(df, ["wins"], 2, 3, q)                      # counters missing
    # item_wins / item_fails scale the item one-hot by the event's own wins / fails columns (fm.py:74-77)
    df2 = df.assign(wins=[0, 1, 1, 0, 0, 0, 0], fails=[0, 0, 1, 0, 1, 0, 0])
    X = ktm.df_to_sparse(df2, ["item_wins", "item_fails"], 2, 3, q).toarray()
    assert X[1, 1] == 1 and X[2, 3 + 1] == 1 and X[4, 3 + 2] == 1 and X.sum() == 4


def test_dataset_layout_roundtrip(tmp_path):
    users, items, outcomes, q = ktm.make_ktm_events(n_events=500, user_num=12, item_num=30, n_skills=5, seed=3)
    assert len(users) == 500 and q.shape == (30, 5) and set(np.unique(outcomes)) <= {0.0, 1.0}
    assert (np.diff(users) >= 0).all()   # a student's events are contiguous
    ktm.write_dataset("syn", users, items, outcomes, q, 12, 30, data_folder=str(tmp_path), batch_size=100)
    df, config, q2, sw, sf = ktm.load_dataset("syn", str(tmp_path))
    assert config == dict(USER_NUM=12, ITEM_NUM=30, NB_CLASSES=2, BATCH_SIZE=100)
    assert df["user"].dtype == np.int32 and df["outcome"].dtype == np.float32 and len(df) == 500
    assert np.array_equal(df["user"], users) and np.array_equal(df["item"], items)
    assert (q2 != q).nnz == 0 and sw.shape == (500, 5)
    legend = dataio.get_legend(dict(d=5, users=True, items=True, skills=True, wins=True, fails=True))
    X = ktm.df_to_sparse(df, legend[3], 12, 30, q2, sw, sf)
    assert X.shape == (500, 12 + 30 + 5 + 5 + 5)
    # all.csv's wins/fails columns: the user's earlier wins / fails on this very item
    k = int(np.flatnonzero((df["wins"] + df["fails"]) > 0)[0])
    prev = df.iloc[:k]
    same = prev[(prev["user"] == df["user"][k]) & (prev["item"] == df["item"][k])]
    assert df["wins"][k] == (same["outcome"] > 0.5).sum() and df["fails"][k] == (same["outcome"] < 0.5).sum()


# ---- CPU: the FM step of the oracle against torch autograd -----------------------------------------------------------
def _fm_problem(rng, F, d, n, max_nnz=5, real_valued=True, min_nnz=1):
    lens = rng.integers(min_nnz, max_nnz + 1, n)
    indptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    p = 1.0 / np.arange(1, F + 1)
    indices = np.concatenate([rng.choice(F, size=k, replace=False, p=p / p.sum()) for k in lens] + [[]]).astype(np.int32)
    data = (rng.integers(1, 4, indptr[-1]) if not real_valued else rng.uniform(0.5, 2.0, indptr[-1])).astype(np.float32)
    return indptr, indices, data


ORACLE_SGD_FLAGS = [oracle.OPT_SGD, oracle.OPT_SGD | oracle.LOSS_SIGMOID_CE, oracle.OPT_SGD | oracle.REG_BIAS]


@pytest.mark.parametrize("flags", ORACLE_SGD_FLAGS)
def test_fm_oracle_gradients_match_torch_autograd(flags):
    """One SGD step of the oracle == var - lr * autograd(cost), cost = data_loss + reg * sum over NON-ZERO OCCURRENCES
    of l2_loss(gathered V row) (+ gathered W with REG_BIAS): the SVD path's per-occurrence L2 (ops.py:81-89,140)."""
    _oracle_sgd_step_vs_autograd(flags, 6)


def _oracle_sgd_step_vs_autograd(flags, d):
    """V's entries are drawn with variance 0.09 * 6 / d, so that the interaction term keeps one scale at every dim."""
    rng = np.random.default_rng(5)
    F, n, lr, reg = 30, 40, 0.01, 0.05
    indptr, indices, data = _fm_problem(rng, F, d, n)
    y = rng.integers(0, 2, n).astype(np.float32)
    w0, W = np.array([0.1], np.float32), rng.normal(0, 0.3, F).astype(np.float32)
    V = rng.normal(0, 0.3 * np.sqrt(6 / d), (F, d)).astype(np.float32)
    orc = oracle.FmOracle(w0, W, V, lr, reg, flags=flags)
    yhat = orc.train_step(indptr, indices, data, y)
    tw0, tW, tV = (torch.tensor(a, dtype=torch.float64, requires_grad=True) for a in (w0, W, V))
    idx = torch.from_numpy(indices.astype(np.int64))
    x = torch.from_numpy(data.astype(np.float64))
    rowof = torch.from_numpy(np.repeat(np.arange(n), np.diff(indptr)))
    Vg, Wg = tV[idx], tW[idx]                      # gathered per non-zero
    xv = Vg * x[:, None]
    s = torch.zeros(n, d, dtype=torch.float64).index_add(0, rowof, xv)
    q = torch.zeros(n, d, dtype=torch.float64).index_add(0, rowof, xv * xv)
    lin = torch.zeros(n, dtype=torch.float64).index_add(0, rowof, Wg * x)
    pred = tw0 + lin + 0.5 * (s * s - q).sum(1)
    ty = torch.from_numpy(y.astype(np.float64))
    if flags & oracle.LOSS_SIGMOID_CE:
        loss = torch.nn.functional.binary_cross_entropy_with_logits(pred, ty, reduction="sum")
    else:
        loss = 0.5 * ((pred - ty) ** 2).sum()
    regul = 0.5 * (Vg ** 2).sum()
    if flags & oracle.REG_BIAS:
        regul = regul + 0.5 * (Wg ** 2).sum()
    (loss + reg * regul).backward()
    np.testing.assert_allclose(yhat, pred.detach().numpy(), rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(orc.V, V - lr * tV.grad.numpy(), rtol=2e-5, atol=2e-6)
    np.testing.assert_allclose(orc.W, W - lr * tW.grad.numpy(), rtol=2e-5, atol=2e-6)
    np.testing.assert_allclose(orc.w0, w0 - lr * tw0.grad.numpy(), rtol=2e-5, atol=2e-6)


def test_fm_oracle_adam_moves_untouched_rows():
    """TF IndexedSlices semantics carried over to the FM: a feature absent from the batch keeps decaying m, v and
    keeps moving while its m != 0."""
    rng = np.random.default_rng(6)
    F, d = 10, 4
    orc = oracle.FmOracle([0.0], np.zeros(F), rng.normal(0, 0.1, (F, d)), 1e-2, 0.01)
    y = np.array([1.0, 0.0], np.float32)
    orc.train_step([0, 2, 4], [0, 1, 2, 3], np.ones(4, np.float32), y)
    V1 = orc.V.copy()
    assert np.array_equal(V1[5:], orc.V[5:]) and orc.slots["m_V"][0].any()
    orc.train_step([0, 2, 4], [4, 5, 6, 7], np.ones(4, np.float32), y)
    assert not np.array_equal(orc.V[0], V1[0])          # row 0 was not in the second batch, yet it moved
    assert np.array_equal(orc.V[8:], V1[8:])            # never-touched rows: m = 0 -> no move
    assert orc.s.global_step == 2


# ---- GPU: the CUDA FM step against the oracle ------------------------------------------------------------------------
def _assert_close(got, ref, what, rtol=RTOL, max_abs=None):
    got, ref = np.asarray(got, np.float64).reshape(-1), np.asarray(ref, np.float64).reshape(-1)
    nref = np.linalg.norm(ref)
    err = np.linalg.norm(got - ref)
    assert err <= rtol * max(nref, 1e-30) + 1e-30, "%s: relative L2 error %.3g" % (what, err / max(nref, 1e-30))
    rms = nref / np.sqrt(max(ref.size, 1))
    bad = np.abs(got - ref) > rtol * np.abs(ref) + rtol * rms + 1e-30
    assert bad.mean() <= 1e-3, "%s: %d of %d entries outside 1e-5" % (what, bad.sum(), ref.size)
    if max_abs is not None:
        assert np.abs(got - ref).max() <= max_abs, what


def _fm_pair(F, d, lr, reg, flags, seed=2, eps=1e-8):
    from tf_recomm_b200.fm_engine import FmEngine
    rng = np.random.default_rng(seed)
    tabs = dict(w0=np.array([0.05], np.float32), W=rng.normal(0, 0.1, F).astype(np.float32),
                V=rng.normal(0, 0.1, (F, d)).astype(np.float32))
    return (FmEngine(F, d, lr, reg, flags=flags, eps=eps, tables=tabs),
            oracle.FmOracle(tabs["w0"], tabs["W"], tabs["V"], lr, reg, flags=flags, eps=eps))


@pytest.mark.gpu
@pytest.mark.parametrize("F,d,n,max_nnz", [(40, 20, 64, 4), (500, 20, 1000, 6), (31028, 20, 10000, 4), (300, 128, 512, 3),
                                           (57, 15, 333, 5), (64, 4, 100, 8)])
@pytest.mark.parametrize("flags", [0, _lib.LOSS_SIGMOID_CE])
def test_fm_train_step_parity_adam(F, d, n, max_nnz, flags):
    """Per-step parameters within 1e-5 relative of the oracle over several steps; yhat from the PRE-update tables."""
    eng, orc = _fm_pair(F, d, 1e-2, 0.01, flags)
    rng = np.random.default_rng(11)
    for step in range(6):
        indptr, indices, data = _fm_problem(rng, F, d, n, max_nnz, real_valued=(step % 2 == 1), min_nnz=0 if step == 3 else 1)
        y = rng.integers(0, 2, n).astype(np.float32)
        yhat = eng.train_step((indptr, indices, data), y).cpu().numpy()
        ref = orc.train_step(indptr, indices, data, y)
        _assert_close(yhat, ref, "yhat step %d" % step)
        got = eng.get_tables()
        for name in ("w0", "W", "V"):
            _assert_close(got[name], getattr(orc, name), "%s step %d" % (name, step), max_abs=4e-2 + 1e-6)
            _assert_close(got["m_" + name], orc.slots["m_" + name], "m_%s step %d" % (name, step))
            _assert_close(got["v_" + name], orc.slots["v_" + name], "v_%s step %d" % (name, step))
    assert eng.global_step == 6 == orc.s.global_step
    assert int((((eng.slot >> 32) & 0xffffffff) == 6).sum()) == 0   # no slot entry carries the next step's stamp


@pytest.mark.gpu
@pytest.mark.parametrize("flags", [_lib.OPT_SGD, _lib.OPT_SGD | _lib.LOSS_SIGMOID_CE | _lib.REG_BIAS])
def test_fm_train_step_parity_sgd(flags):
    eng, orc = _fm_pair(200, 20, 1e-3, 0.01, flags)
    rng = np.random.default_rng(12)
    for step in range(5):
        indptr, indices, data = _fm_problem(rng, 200, 20, 400, 5)
        y = rng.integers(0, 2, 400).astype(np.float32)
        yhat = eng.train_step((indptr, indices, data), y).cpu().numpy()
        _assert_close(yhat, orc.train_step(indptr, indices, data, y), "yhat")
        got = eng.get_tables()
        for name in ("w0", "W", "V"):
            _assert_close(got[name], getattr(orc, name), "%s step %d" % (name, step))


@pytest.mark.gpu
def test_fm_hot_feature_and_two_hot_rows_equal_svd_step():
    """(1) a feature present in EVERY row (a run of n occurrences crossing many 32-entry tiles); (2) on (user | item)
    two-hot rows the FM step is the SVD step (forward.py:47-61 builds exactly such rows): compare with SvdEngine."""
    from tf_recomm_b200 import init
    from tf_recomm_b200.engine import SvdEngine
    from tf_recomm_b200.fm_engine import FmEngine
    rng = np.random.default_rng(13)
    F, d, n = 50, 20, 3000
    eng, orc = _fm_pair(F, d, 1e-2, 0.01, 0)
    lens = np.full(n, 3)
    indptr = np.arange(0, 3 * n + 1, 3, dtype=np.int64)
    indices = np.stack([np.zeros(n, np.int64), rng.integers(1, 25, n), rng.integers(25, F, n)], 1).reshape(-1).astype(np.int32)
    data = np.ones(3 * n, np.float32)
    y = rng.integers(0, 2, n).astype(np.float32)
    for _ in range(3):
        _assert_close(eng.train_step((indptr, indices, data), y).cpu().numpy(), orc.train_step(indptr, indices, data, y), "yhat")
    _assert_close(eng.get_tables()["V"], orc.V, "V with a hot feature", rtol=2e-5)
    assert lens.sum() == len(indices)
    U, I, d, B = 60, 40, 20, 500
    tabs = init.init_tables(U, I, d, seed=4)
    svd = SvdEngine(U, I, d, 1e-2, 0.05, tables=tabs)
    fm = FmEngine(U + I, d, 1e-2, 0.05, tables=dict(w0=tabs["mu"], W=np.concatenate([tabs["user_bias"], tabs["item_bias"]]),
                                                    V=np.concatenate([tabs["user_feat"], tabs["item_feat"]])))
    for _ in range(4):
        users, items = rng.integers(0, U, B).astype(np.int32), rng.integers(0, I, B).astype(np.int32)
        rates = rng.integers(1, 6, B).astype(np.float32)
        lg, _ = svd.train_step(users, items, rates)
        yh = fm.train_step((np.arange(0, 2 * B + 1, 2), np.stack([users, U + items], 1).reshape(-1), np.ones(2 * B, np.float32)), rates)
        np.testing.assert_allclose(yh.cpu().numpy(), lg.cpu().numpy(), rtol=1e-4, atol=1e-5)
    ts, tf_ = svd.get_tables(), fm.get_tables()
    np.testing.assert_allclose(tf_["V"][:U], ts["user_feat"], rtol=1e-3, atol=1e-5)
    np.testing.assert_allclose(tf_["V"][U:], ts["item_feat"], rtol=1e-3, atol=1e-5)
    np.testing.assert_allclose(tf_["W"][:U], ts["user_bias"], rtol=1e-3, atol=1e-5)
    np.testing.assert_allclose(tf_["w0"], ts["mu"], rtol=1e-3, atol=1e-5)


@pytest.mark.gpu
def test_fm_graph_epoch_equals_eager_epoch_and_learns():
    """run_epoch with captured graphs == the same steps launched eagerly (bit-identical); training on a planted KTM
    dataset (config[2] shape family, reduced) lowers the held-out log-loss below the constant predictor's."""
    from tf_recomm_b200.fm_engine import FmEngine
    users, items, outcomes, q = ktm.make_ktm_events(n_events=20000, user_num=300, item_num=800, n_skills=20, seed=5)
    import pandas as pd
    df = pd.DataFrame(dict(user=users, item=items, outcome=outcomes, wins=0, fails=0))
    X = ktm.df_to_sparse(df, ["users", "items", "skills"], 300, 800, q)
    n_tr = 16000
    perm = np.random.default_rng(0).permutation(len(df))
    tr, te = perm[:n_tr], perm[n_tr:]
    engs = [FmEngine(X.shape[1], 20, 1e-2, 3e-2, flags=_lib.LOSS_SIGMOID_CE, seed=1) for _ in range(2)]
    chunks = np.array_split(tr, 8)
    for e, eng in enumerate(engs):
        batches = [eng.upload_csr(X[c], outcomes[c]) for c in chunks]
        for _ in range(6):
            eng.run_epoch(batches, use_graph=(e == 0))
    a, b = engs[0].get_tables(), engs[1].get_tables()
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    assert engs[0].global_step == 6 * 8
    p = torch.sigmoid(engs[0].forward(X[te]).double()).cpu().numpy().clip(1e-7, 1 - 1e-7)
    yt = outcomes[te]
    nll = -np.mean(yt * np.log(p) + (1 - yt) * np.log(1 - p))
    base = yt.mean()
    nll0 = -np.mean(yt * np.log(base) + (1 - yt) * np.log(1 - base))
    assert nll < 0.95 * nll0, (nll, nll0)


@pytest.mark.gpu
def test_fm_driver_end_to_end(tmp_path):
    """`python fm.py --dataset syn --d 5 --users --items --skills --iter 20 --synthetic 4000`: the reference's outputs."""
    import fm as fm_driver
    res = fm_driver.main(["--dataset", "syn", "--d", "5", "--users", "--items", "--skills", "--iter", "20", "--synthetic",
                          "4000", "--data_folder", str(tmp_path), "--seed", "0", "--folds", "2", "--batch", "500"])
    folder = os.path.join(str(tmp_path), "syn", "uis5")
    for run in ("0", "1"):
        r = json.load(open(os.path.join(folder, run, "results.json")))
        assert set(r["metrics"]) == {"ACC", "AUC", "NLL"} and r["legends"]["short"] == "uis5"
        assert os.path.exists(os.path.join(folder, run, "vectors-5.npy"))
    assert os.path.exists(os.path.join(folder, "X.npz"))
    assert all(0.5 < r["AUC"] <= 1.0 for r in res), res   # held-out USERS: only item / skill effects transfer
