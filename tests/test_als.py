"""Alternating least squares on the device: tfr_als_half_sweep / tfr_svd_objective (csrc/als.cu), SvdEngine.als_data /
als_sweep / training_objective above them, and svd_train_val.py --solver als.  The numpy reference below is one
np.linalg.solve per row; it is pinned to the training step's own gradients (oracle/np_oracle.py::grads)."""
import io
import os
import re
import subprocess
from contextlib import redirect_stdout

import numpy as np
import pytest

from oracle import np_oracle
from test_fold_in import fold_ref
from tf_recomm_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NVCC = "/usr/local/cuda/bin/nvcc"
ALS_FLAGS = [0, _lib.REG_BIAS]


# ---- numpy float64 reference -------------------------------------------------------------------------------------------------
def half_ref(Fx, fb, mu, rows, partner, rates, n_rows, reg, flags):
    """Every row r in [0, n_rows) solved against the fixed side (Fx, fb): fold-in's system over the ratings with
    rows == r (x = [Fx[partner] ; 1], target r - mu - fb[partner]).  -> [n_rows, d + 1] float64."""
    out = np.zeros((n_rows, Fx.shape[1] + 1))
    order = np.argsort(rows, kind="stable")
    starts = np.searchsorted(rows[order], np.arange(n_rows + 1))
    for r in range(n_rows):
        sel = order[starts[r]:starts[r + 1]]
        out[r] = fold_ref(Fx, fb, mu, partner[sel], rates[sel], reg, flags)
    return out


def residuals(T, users, items, rates):
    """e = r - mu - b_u - b_i - p_u.q_i in float64 from the tables T."""
    f = {k: np.asarray(v, np.float64) for k, v in T.items()}
    dot = np.einsum("nd,nd->n", f["user_feat"][users], f["item_feat"][items])
    return rates.astype(np.float64) - f["mu"].reshape(-1)[0] - f["user_bias"][users] - f["item_bias"][items] - dot


def loss(T, users, items, rates, reg, flags):
    f = {k: np.asarray(v, np.float64) for k, v in T.items()}
    e = residuals(T, users, items, rates)
    pen = (f["user_feat"][users] ** 2).sum() + (f["item_feat"][items] ** 2).sum()
    if flags & _lib.REG_BIAS:
        pen += (f["user_bias"][users] ** 2).sum() + (f["item_bias"][items] ** 2).sum()
    return 0.5 * (e @ e) + 0.5 * float(np.float32(reg)) * pen


# ---- CPU -------------------------------------------------------------------------------------------------------------------
def _small_problem(seed):
    rng = np.random.default_rng(seed)
    U, I, d = 11, 9, 5
    p = dict(mu=np.array([3.2], np.float32), user_bias=rng.normal(0, 0.3, U).astype(np.float32),
             item_bias=rng.normal(0, 0.3, I).astype(np.float32), user_feat=rng.normal(0, 0.3, (U, d)).astype(np.float32),
             item_feat=rng.normal(0, 0.3, (I, d)).astype(np.float32))
    n = 120
    users, items = rng.integers(0, U - 1, n), rng.integers(0, I - 1, n)   # the last user and item have no ratings
    users[:5], items[:5] = users[5], items[5]                               # duplicates
    return p, users, items, rng.integers(1, 6, n).astype(np.float32), U, I, d


@pytest.mark.parametrize("flags", ALS_FLAGS)
def test_reference_sweep_zeroes_each_blocks_training_gradients(flags):
    """After each block of the numpy sweep, that block's training gradients (the oracle's per-occurrence gradients summed
    per row, duplicates included) vanish; a perturbed row's do not."""
    p, users, items, rates, U, I, d = _small_problem(flags)
    reg, rb = np.float32(0.05), bool(flags & _lib.REG_BIAS)

    def g():
        return np_oracle.grads(p, users, items, rates, reg, reg_bias=rb)

    def row_sums(vals, ids, n):
        out = np.zeros((n,) + vals.shape[1:])
        np.add.at(out, ids, vals.astype(np.float64))
        return out
    th = half_ref(p["item_feat"], p["item_bias"], p["mu"][0], users, items, rates, U, reg, flags)
    p["user_feat"][:], p["user_bias"][:] = th[:, :d], th[:, d]
    gr = g()
    assert np.abs(row_sums(gr["g_uf"], users, U)).max() < 1e-5 * 5 and np.abs(row_sums(gr["g_ub"], users, U)).max() < 1e-5 * 5
    assert not p["user_feat"][U - 1].any() and p["user_bias"][U - 1] == 0
    th = half_ref(p["user_feat"], p["user_bias"], p["mu"][0], items, users, rates, I, reg, flags)
    p["item_feat"][:], p["item_bias"][:] = th[:, :d], th[:, d]
    gr = g()
    assert np.abs(row_sums(gr["g_if"], items, I)).max() < 1e-5 * 5 and np.abs(row_sums(gr["g_ib"], items, I)).max() < 1e-5 * 5
    p["mu"][0] = np.float32(p["mu"][0] + residuals(p, users, items, rates).mean())
    assert abs(float(g()["g_mu"])) < 1e-4 * len(users)
    # a perturbed item row: the test has teeth
    p["item_bias"][2] += 0.1
    assert np.abs(row_sums(g()["g_ib"], items, I)[2]) > 1e-2


def _half(L, dim=16, flags=0, var_mask=_lib.VAR_ALL, reg=0.05, n_light=3, n_heavy=1, n_chunks=2, feat=1, fixed=1,
          failed=1, ws=1, ws_bytes=1 << 30, chunk=64):
    """tfr_als_half_sweep with dummy (never dereferenced) pointers: only the argument checks can run."""
    p = 4096
    return L.tfr_als_half_sweep(fixed and p, p, p, 100, dim, 0, flags, var_mask, reg, p, p, p, p, n_light, p, p, n_heavy,
                                p, n_chunks, chunk, feat and p, 0, p, failed and p, ws and p, ws_bytes, None)


def test_invalid_arguments_are_refused_before_any_cuda_call():
    L = _lib.load()
    for kw in (dict(flags=_lib.LOSS_SIGMOID_CE), dict(flags=_lib.ABS_ITEM), dict(flags=_lib.FORK_FLAGS),
               dict(var_mask=_lib.VAR_UF), dict(var_mask=_lib.VAR_ALL & ~_lib.VAR_MU), dict(dim=129), dict(dim=0),
               dict(reg=0.0), dict(reg=-1.0), dict(reg=float("nan")), dict(reg=float("inf")), dict(feat=0), dict(fixed=0),
               dict(failed=0), dict(ws=0), dict(chunk=0), dict(n_chunks=0)):
        assert _half(L, **kw) == -1, kw   # TFR_ERR_INVALID
    assert _half(L, ws_bytes=100) == -3   # TFR_ERR_WORKSPACE, still before any CUDA call
    assert _half(L, n_light=0, n_heavy=0, n_chunks=0, feat=0, fixed=0, failed=0, ws=0) == 0   # nothing to solve: a no-op
    p = 4096
    obj = lambda flags=0, out=p, mu_out=0, ws=p, reg=0.05: L.tfr_svd_objective(  # noqa: E731
        p, p, p, p, p, 10, 10, 8, 0, 0, flags, reg, p, p, p, p, out, mu_out, ws, 1 << 20, None)
    for kw in (dict(flags=_lib.LOSS_SIGMOID_CE), dict(out=0), dict(ws=0), dict(reg=-1.0), dict(reg=float("nan"))):
        assert obj(**kw) == -1, kw


def test_workspace_and_chunk_knob():
    L = _lib.load()
    D = 129
    assert L.tfr_als_workspace_bytes(1, 128) >= (D * (D + 1) // 2 + D) * 8 == 68112
    assert L.tfr_als_workspace_bytes(1000, 128) >= 1000 * 68112
    assert L.tfr_als_workspace_bytes(-1, 8) < 0 and L.tfr_als_workspace_bytes(1, 129) < 0
    old = _lib.tune_get("ALS_CHUNK")
    try:
        for v, want in ((1, 32), (0, 32), (33, 64), (4096, 4096), (1 << 30, 1 << 20)):
            _lib.tune_set("ALS_CHUNK", v)
            assert L.tfr_als_chunk() == want, v
    finally:
        _lib.tune_set("ALS_CHUNK", old)


@pytest.mark.skipif(not os.path.exists(NVCC), reason="needs the CUDA toolkit")
def test_als_kernels_compile_without_spills(tmp_path):
    from test_rank_users import _ptxas_lines
    info = {}
    for src in ("als.cu", "fold_in.cu"):
        obj, log = str(tmp_path / (src + ".o")), str(tmp_path / (src + ".txt"))
        with open(log, "w") as f:
            subprocess.check_call([NVCC, "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-ccbin",
                                   "/usr/bin/g++", "-Xcompiler", "-fPIC", "-Xptxas", "-v", "-c",
                                   os.path.join(ROOT, "tf-recomm_b200", "csrc", src), "-o", obj],
                                  stdout=f, stderr=subprocess.STDOUT)
        info.update(_ptxas_lines(log))
    half_sweep = ["void tfr::half_sweep_%s_kernel<tfr::FiForm<true, false, true> >" % k   # FiRatings
                  for k in ("rows", "chunk_gram", "heavy_solve")]
    names = {*half_sweep, "tfr::als_objective_rows_kernel", "tfr::als_objective_finish_kernel", "tfr::fold_in_kernel"}
    assert names <= set(info), sorted(info)
    for name in names:
        regs, stack, st, ld = info[name]
        assert (stack, st, ld) == (0, 0, 0), (name, info[name])
    for name in (*half_sweep, "tfr::fold_in_kernel"):
        assert info[name][0] <= 128, (name, info[name])   # __launch_bounds__(256, 2): two CTAs per SM


# ---- GPU -------------------------------------------------------------------------------------------------------------------
def _ratings(U, I, d, seed):
    """Users 0..5 rate 0, 1, d, d + 1, d + 2 and 3000 filler items (>= 8); items 0..5 are rated 0, 1, d, d + 1, d + 2 and
    5000 times by filler users (>= 8); the fillers also rate each other (about 60 ratings each).  Duplicates in every
    controlled row."""
    rng = np.random.default_rng(seed)
    us, its = [], []
    for k, (cu, ci) in enumerate(zip([0, 1, d, d + 1, d + 2, 3000], [0, 1, d, d + 1, d + 2, 5000])):
        f = rng.integers(8, I, cu)
        if cu >= 2:
            f[-1] = f[0]
        us.append(np.full(cu, k)); its.append(f)
        g = rng.integers(8, U, ci)
        if ci >= 2:
            g[-1] = g[0]
        us.append(g); its.append(np.full(ci, k))
    n_fill = 12000
    us.append(rng.integers(8, U, n_fill)); its.append(rng.integers(8, I, n_fill))
    users, items = np.concatenate(us), np.concatenate(its)
    perm = rng.permutation(len(users))
    rates = rng.integers(1, 6, len(users)).astype(np.float32)
    return users[perm].astype(np.int32), items[perm].astype(np.int32), rates


def _engine(U, I, d, flags=0, seed=5, reg=0.05):
    from tf_recomm_b200 import init
    from tf_recomm_b200.engine import SvdEngine
    tabs = init.init_tables(U, I, d, seed=seed, bias_init="truncated_normal")
    tabs["user_feat"] *= 10
    tabs["item_feat"] *= 10
    tabs["mu"][:] = 3.5
    return SvdEngine(U, I, d, 1e-3, reg, flags=flags, tables=tabs)


def _tables(eng):
    return {n: eng.t[n].cpu().numpy().copy() for n in ("mu", "user_bias", "item_bias", "user_feat", "item_feat")}


def _user_half(eng, data, reg):
    import torch
    T = eng.t
    with torch.cuda.device(eng.device):
        eng._half_sweep(data, reg, data.by_user, data.user_plan, (T["item_feat"], T["item_bias"], eng.I),
                        (T["user_feat"], T["user_bias"]))


def _item_half(eng, data, reg):
    import torch
    T = eng.t
    with torch.cuda.device(eng.device):
        eng._half_sweep(data, reg, data.by_item, data.item_plan, (T["user_feat"], T["user_bias"], eng.U),
                        (T["item_feat"], T["item_bias"]))


def _mu_step(eng, data, reg):
    import torch
    with torch.cuda.device(eng.device):
        eng._objective(data, reg, eng.t["mu"].data_ptr())


def _check_rows(got_feat, got_bias, ref):
    got = np.hstack([got_feat.astype(np.float64), got_bias.astype(np.float64)[:, None]])
    for r in range(len(ref)):
        tol = 2.0 ** -24 * np.abs(ref[r]) + 1e-10 * np.abs(ref[r]).max()
        assert (np.abs(got[r] - ref[r]) <= tol).all(), (r, np.abs(got[r] - ref[r]).max(), np.abs(ref[r]).max())


def _half_steps_against_numpy(eng, users, items, rates, reg, flags):
    data = eng.als_data(users, items, rates)
    T0 = _tables(eng)
    _user_half(eng, data, reg)
    T1 = _tables(eng)
    ref = half_ref(T0["item_feat"], T0["item_bias"], T0["mu"][0], users, items, rates, eng.U, reg, flags)
    _check_rows(T1["user_feat"], T1["user_bias"], ref)
    assert all(np.array_equal(T0[n], T1[n]) for n in ("mu", "item_feat", "item_bias"))
    _item_half(eng, data, reg)
    T2 = _tables(eng)
    ref = half_ref(T1["user_feat"], T1["user_bias"], T1["mu"][0], items, users, rates, eng.I, reg, flags)
    _check_rows(T2["item_feat"], T2["item_bias"], ref)
    assert all(np.array_equal(T1[n], T2[n]) for n in ("mu", "user_feat", "user_bias"))
    _mu_step(eng, data, reg)
    T3 = _tables(eng)
    assert T3["mu"][0] == np.float32(T2["mu"][0] + residuals(T2, users, items, rates).mean())
    assert int(data.failed.item()) == 0
    return data


@pytest.mark.gpu
@pytest.mark.parametrize("d", [1, 15, 32, 64, 128])
@pytest.mark.parametrize("flags", ALS_FLAGS)
@pytest.mark.parametrize("sgd", [False, True])
def test_half_steps_match_numpy(d, flags, sgd):
    """Each half-step against np.linalg.solve from the GPU's own tables just before it: every entry within fold-in's bound
    2^-24 |ref| + 1e-10 max|ref|, for rows with 0, 1, d, d + 1, d + 2 and thousands of ratings; mu = fl32(mu + mean e)."""
    U, I = 300, 200
    users, items, rates = _ratings(U, I, d, seed=d + flags)
    eng = _engine(U, I, d, flags=flags | (_lib.OPT_SGD if sgd else 0))
    data = _half_steps_against_numpy(eng, users, items, rates, 0.05, flags)
    assert data.item_plan.heavy.numel() == 1 and data.chunk == _lib.tune_get("ALS_CHUNK")   # the 5000-rating item splits


@pytest.mark.gpu
def test_split_path_meets_the_bound_and_keeps_its_bits():
    """ALS_CHUNK at its minimum: most rows split, they meet the same bound, and the bits are the same run to run, between
    two engines and between an eager sweep and a CUDA-graph replay of it."""
    import torch
    U, I, d, reg = 300, 200, 32, 0.05
    users, items, rates = _ratings(U, I, d, seed=77)
    old = _lib.tune_get("ALS_CHUNK")
    try:
        _lib.tune_set("ALS_CHUNK", 1)
        eng = _engine(U, I, d, flags=_lib.REG_BIAS)
        data = _half_steps_against_numpy(eng, users, items, rates, reg, _lib.REG_BIAS)
        assert data.chunk == 32
        cnt_u = np.bincount(users, minlength=U)
        assert data.user_plan.heavy.numel() == (cnt_u > 32).sum() > U // 2
        start = _tables(eng)

        def sweep_from_start(e, dat):
            for n, a in start.items():
                e.t[n].copy_(torch.from_numpy(a.reshape(e.t[n].shape)))
            e.als_sweep(dat, reg=reg)
            torch.cuda.synchronize(e.device)
            return [v.view(np.uint8) for v in _tables(e).values()]
        first = sweep_from_start(eng, data)
        assert all(np.array_equal(a, b) for a, b in zip(first, sweep_from_start(eng, data)))
        eng2 = _engine(U, I, d, flags=_lib.REG_BIAS, seed=9)
        data2 = eng2.als_data(users, items, rates)
        assert all(np.array_equal(a, b) for a, b in zip(first, sweep_from_start(eng2, data2)))
        # graph: capture one sweep, replay it from the start
        for n, a in start.items():
            eng.t[n].copy_(torch.from_numpy(a.reshape(eng.t[n].shape)))
        exe = eng._capture(lambda: eng.als_sweep(data, reg=reg))
        try:
            for n, a in start.items():
                eng.t[n].copy_(torch.from_numpy(a.reshape(eng.t[n].shape)))
            _lib.check(eng.L.tfr_graph_launch(exe, torch.cuda.current_stream(eng.device).cuda_stream))
            torch.cuda.synchronize(eng.device)
            assert all(np.array_equal(a, b) for a, b in zip(first, [v.view(np.uint8) for v in _tables(eng).values()]))
        finally:
            eng.L.tfr_graph_destroy(exe)
    finally:
        _lib.tune_set("ALS_CHUNK", old)


@pytest.mark.gpu
@pytest.mark.parametrize("sgd", [False, True])
def test_user_half_sweep_equals_fold_in_bit_for_bit(sgd):
    U, I, d = 300, 200, 64
    users, items, rates = _ratings(U, I, d, seed=3)
    eng = _engine(U, I, d, flags=_lib.OPT_SGD if sgd else 0)
    data = eng.als_data(users, items, rates)
    assert data.user_plan.heavy.numel() == 0
    f = eng.fold_in(users, items, rates, n=U, reg=0.05)
    _user_half(eng, data, 0.05)
    assert np.array_equal(f.feat.cpu().numpy().view(np.uint32), eng.t["user_feat"].cpu().numpy().view(np.uint32))
    assert np.array_equal(f.bias.cpu().numpy().view(np.uint32), eng.t["user_bias"].cpu().numpy().view(np.uint32))


def _train_split(ratings=None):
    from tf_recomm_b200 import config, synthetic
    U, I, N = synthetic.SHAPES["ml1m"]
    au, ai, ar = synthetic.make_ratings(U, I, ratings or N, seed=config.SEED)
    (tu, ti, tr), (vu, vi, vr) = synthetic.split(au, ai, ar)
    return U, I, (tu, ti, tr), (vu, vi, vr)


@pytest.mark.gpu
def test_objective_never_rises_over_ten_sweeps():
    """ML-1M shape, d = 15, the driver's initialisation: every half-step and every mu step gives L_after <= L_before
    (1 + 1e-9), and the objective matches numpy's."""
    from tf_recomm_b200 import config, init
    from tf_recomm_b200.engine import SvdEngine
    U, I, (tu, ti, tr), _ = _train_split()
    reg = config.LAMBDA_REG
    eng = SvdEngine(U, I, 15, config.LEARNING_RATE, reg, tables=init.init_tables(U, I, 15, seed=13575))
    data = eng.als_data(tu, ti, tr)
    obj = eng.training_objective(data)
    want = loss(_tables(eng), tu, ti, tr, reg, 0)
    assert abs(obj["loss"] - want) <= 1e-9 * want and obj["n"] == len(tu)
    assert abs(obj["rmse"] - np.sqrt(np.mean(residuals(_tables(eng), tu, ti, tr) ** 2))) < 1e-12
    first, prev = obj["loss"], obj["loss"]
    for _ in range(10):
        for step in (_user_half, _item_half, _mu_step):
            step(eng, data, reg)
            cur = eng.training_objective(data)["loss"]
            assert cur <= prev * (1 + 1e-9), (step.__name__, prev, cur)
            prev = cur
    assert prev < first
    assert abs(prev - loss(_tables(eng), tu, ti, tr, reg, 0)) <= 1e-9 * prev


@pytest.mark.gpu
def test_sweep_leaves_the_optimizer_state_and_adam_continues():
    import oracle
    U, I, d = 300, 200, 16
    users, items, rates = _ratings(U, I, d, seed=12)
    eng = _engine(U, I, d)
    rng = np.random.default_rng(4)
    B = 500
    for _ in range(2):   # some Adam state first
        eng.train_step(rng.integers(0, U, B), rng.integers(0, I, B), rng.integers(1, 6, B).astype(np.float32))
    snap = lambda: [a.cpu().numpy().copy() for a in (eng.slots["m_user_feat"], eng.slots["v_user_feat"],  # noqa: E731
                                                     eng.slots["m_item_feat"], eng.slots["v_item_feat"],
                                                     *(eng.slots[k] for k in sorted(eng.slots) if "feat" not in k),
                                                     eng.user_slot, eng.item_slot, eng.opt)]
    before = snap()
    data = eng.als_data(users, items, rates)
    assert int(eng.als_sweep(data).item()) == 0
    after = snap()
    assert all(np.array_equal(a.view(np.uint8), b.view(np.uint8)) for a, b in zip(before, after))
    # Adam from the ALS tables, against the oracle stepped from the same tables and optimizer state
    tabs = eng.get_tables()
    s = eng.opt_scalars()
    orc = oracle.SvdOracle(tabs["mu"], tabs["user_bias"], tabs["item_bias"], tabs["user_feat"], tabs["item_feat"], 1e-3,
                           0.05)
    for k, v in orc.slots.items():   # in place: the oracle's state struct points at these arrays
        v[...] = tabs[k].reshape(v.shape)
    orc.s.beta1_power, orc.s.beta2_power, orc.s.global_step = s.beta1_power, s.beta2_power, s.global_step
    for _ in range(2):
        bu, bi = rng.integers(0, U, B).astype(np.int32), rng.integers(0, I, B).astype(np.int32)
        br = rng.integers(1, 6, B).astype(np.float32)
        logits, _ = eng.train_step(bu, bi, br)
        ref_logits, _ = orc.train_step(bu, bi, br)
        np.testing.assert_allclose(logits.cpu().numpy(), ref_logits, rtol=1e-5, atol=1e-6)
    got = eng.get_tables()
    for n in ("mu", "user_bias", "item_bias", "user_feat", "item_feat"):
        np.testing.assert_allclose(got[n].reshape(getattr(orc, n).shape), getattr(orc, n), rtol=1e-5, atol=2e-7)


@pytest.mark.gpu
def test_unsupported_models_are_refused():
    from tf_recomm_b200.engine import SvdEngine, TfrError
    users, items, rates = np.array([0, 1]), np.array([1, 0]), np.array([3.0, 4.0], np.float32)
    for kw in (dict(flags=_lib.ABS_ITEM), dict(flags=_lib.LOSS_SIGMOID_CE), dict(flags=_lib.FORK_FLAGS),
               dict(var_mask=_lib.VAR_UF | _lib.VAR_UB), dict(d=129)):
        d = kw.pop("d", 8)
        eng = SvdEngine(4, 4, d, 1e-3, 0.05, **kw)
        with pytest.raises(TfrError):
            eng.als_data(users, items, rates)
    eng = SvdEngine(4, 4, 8, 1e-3, 0.05)
    data = eng.als_data(users, items, rates)
    for reg in (0.0, -1.0, float("nan"), float("inf")):
        with pytest.raises(TfrError):
            eng.als_sweep(data, reg=reg)
    with pytest.raises(TfrError):
        eng.als_data([0, 4], [1, 0], [3.0, 4.0])


@pytest.mark.gpu
def test_driver_als(tmp_path):
    import recommend
    import svd_train_val
    from tf_recomm_b200 import synthetic
    from tf_recomm_b200.engine import SvdEngine
    ckpt = str(tmp_path / "als.ckpt")
    data = ["--synthetic", "ml1m", "--ratings", "100000"]
    buf = io.StringIO()
    with redirect_stdout(buf):
        svd_train_val.main(data + ["--solver", "als", "--epochs", "3", "--dim", "15", "--checkpoint", ckpt, "--logdir",
                                   str(tmp_path / "log"), "--topk", "10"])
    lines = [ln for ln in buf.getvalue().splitlines() if "TRAIN(" in ln]
    assert len(lines) == 3, buf.getvalue()
    train = [float(re.search(r"TRAIN\(size=(\d+)/(\d+), rmse=([0-9.]+)\)", ln).group(3)) for ln in lines]
    sizes = [re.search(r"TRAIN\(size=(\d+)/(\d+)", ln).groups() for ln in lines]
    assert all(a == b for a, b in sizes)
    assert all(b <= a for a, b in zip(train, train[1:])), train
    assert buf.getvalue().count("TOPK(k=10") == 3
    eng = SvdEngine.from_checkpoint(ckpt)
    assert (eng.U, eng.I, eng.d) == (*synthetic.SHAPES["ml1m"][:2], 15)
    out = io.StringIO()
    recommend.main(["--checkpoint", ckpt, "--users", "3,7", "--k", "5"] + data, out=out)
    assert [ln.split("\t")[0] for ln in out.getvalue().splitlines()] == ["3", "7"]
    with pytest.raises(SystemExit):
        svd_train_val.main(data + ["--solver", "als", "--variant", "fork", "--epochs", "1"])
