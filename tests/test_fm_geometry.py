"""The FM forward and train step at every dim up to 512 and every tuning knob.

tfr_fm_forward (csrc/fm.cu) runs one of the (VEC, L, UNITS) instantiations of fm_forward_kernel listed in TFR_FM_CASES:
(VEC, L) is row_geom's and UNITS = ceil(dim / VEC / L) rounded up to 1, 2, 4, 8 or 16.  The FM step's gradient sums run
the generic unfused segment-sum kernel at seg_geom's geometry (tests/test_geometry.py mirrors both).  The CPU tests read the
list out of fm.cu, mirror the dispatch, check that every dim of 1..512 has an instantiation and that the GPU sweeps reach
every forward and segment-sum instantiation, and check the C oracle's FM against float64 at dims up to 512.  The GPU tests
compare the forward and the step with the oracle at every sweep dim and under the segment-sum knobs, and the step under
the geometry-only knobs with a default-knob run, bit for bit.
"""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest
import scipy.sparse as sp

import oracle
from oracle import np_oracle
from test_geometry import (BIT_SETTINGS, KNOB_DIMS, KNOBS, NVCC, SEG_TILES, SEG_UNITS, SWEEP_DIMS, row_geom, seg_cases,
                           seg_geom, tuned)
from test_ktm_fm import ORACLE_SGD_FLAGS, RTOL, _assert_close, _fm_pair, _fm_problem, _oracle_sgd_step_vs_autograd
from tf_recomm_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FM_CU = os.path.join(ROOT, "tf-recomm_b200", "csrc", "fm.cu")

# the dim sweep of the FM: test_geometry's (every seg_geom case of the default geometry, every row_geom pair) and dims
# whose forward rounds its unit count up (67, 95: 3 -> 4 scalar units, 300: 3 -> 4 float4 units, 130: 5 -> 8)
FM_DIMS = sorted(set(SWEEP_DIMS) | {65, 67, 95, 130, 300, 384})
# the forward's instantiations when it dispatched on the exact unit count: every dim that ran then keeps its kernel
FM_CASES_EXACT_UNITS = {(4, 1, 1), (4, 2, 1), (4, 4, 1), (4, 8, 1), (4, 16, 1), (4, 32, 1), (4, 32, 2), (4, 32, 4),
                        (1, 1, 1), (1, 2, 1), (1, 4, 1), (1, 8, 1), (1, 16, 1), (1, 32, 1), (1, 32, 2), (1, 32, 4)}
FM_MODELS = {"adam_se": 0, "adam_ce": _lib.LOSS_SIGMOID_CE,
             "sgd_ce_regbias": _lib.OPT_SGD | _lib.LOSS_SIGMOID_CE | _lib.REG_BIAS}
ORACLE_DIMS = [1, 20, 256, 257, 300, 384, 511, 512]
U24 = 2.0 ** -24   # fp32 unit roundoff


# ---- Python mirror of the forward's dispatch -------------------------------------------------------------------------------
def fm_cases():
    """The (VEC, L, UNITS) list of TFR_FM_CASES in csrc/fm.cu."""
    src = open(FM_CU).read()
    cases = [tuple(int(x) for x in m) for m in re.findall(r"\b(?:X|TFR_FM_CASE)\((\d+), (\d+), (\d+)\)", src)]
    assert len(cases) == len(set(cases))
    return set(cases)


def _exact_units(dim):
    vec, lanes = row_geom(dim)
    return vec, lanes, -(-(dim // vec) // lanes)


def fm_geom(dim):
    """fm.cu: the (VEC, L, UNITS) tfr_fm_forward launches for dim."""
    vec, lanes, u = _exact_units(dim)
    return vec, lanes, next((r for r in (1, 2, 4, 8, 16) if u <= r), u)


@pytest.fixture(scope="module", autouse=True)
def _restore_knobs():
    """Whatever a test of this module does, every knob it can touch leaves the module as it came in."""
    saved = {k: _lib.tune_get(k) for k in KNOBS}
    try:
        yield
    finally:
        for k, v in saved.items():
            _lib.tune_set(k, v)


# ---- CPU: the dispatch -------------------------------------------------------------------------------------------------------
def test_every_dim_up_to_512_has_an_fm_forward_instantiation():
    cases = fm_cases()
    assert len(cases) == 18
    missing = [d for d in range(1, 513) if fm_geom(d) not in cases]
    assert not missing, missing
    assert fm_geom(513) not in cases and fm_geom(516) not in cases


def test_dims_that_ran_keep_their_instantiation():
    """Rounding the unit count up only gives a kernel to dims that had none: 344 of 1..512 (65..95 with dim % 4 != 0,
    multiples of 4 from 260 to 384, and every dim of 129..511 with dim % 4 != 0).  Every other dim, d = 20 (bench.py's
    also_fm) among them, launches the instantiation it launched before."""
    kept = [d for d in range(1, 513) if _exact_units(d) in FM_CASES_EXACT_UNITS]
    assert 512 - len(kept) == 344
    assert [d for d in kept if fm_geom(d) != _exact_units(d)] == []
    assert fm_geom(20) == (4, 8, 1)


def test_fm_sweeps_reach_every_instantiation():
    """FM_DIMS reach every forward instantiation and every segment-sum geometry any dim reaches by default; with
    test_geometry's SEG_MAX_UNITS sweep they reach every case of the (generic, unfused) segment-sum kernel the FM runs."""
    assert {fm_geom(d) for d in FM_DIMS} == fm_cases(), sorted(fm_cases() - {fm_geom(d) for d in FM_DIMS})
    by_default = {seg_geom(d) for d in FM_DIMS}
    assert by_default == {seg_geom(d) for d in range(1, 513)}, sorted({seg_geom(d) for d in range(1, 513)} - by_default)
    forced = {seg_geom(d, u) for d in KNOB_DIMS for u in SEG_UNITS}
    assert by_default | forced == seg_cases(), sorted(seg_cases() - by_default - forced)


def test_fm_dims_outside_1_to_512_are_refused_before_any_cuda_call():
    """Dummy (never dereferenced) pointers: only the argument checks can run."""
    L = _lib.load()
    p = 4096
    for dim in (0, -1, 513, 516, 1024):
        for n_rows in (0, 10):
            assert L.tfr_fm_forward(n_rows, p, p, p, p, p, p, dim, p, p, None) == -1, (dim, n_rows)   # TFR_ERR_INVALID
        assert b"1 to 512" in L.tfr_last_error(), L.tfr_last_error()
        for sgd in (0, _lib.OPT_SGD):
            t = _lib.FmTables(n_feat=100, dim=dim, w0=p, W=p, V=p, m_w0=p, v_w0=p, m_W=p, v_W=p, m_V=p, v_V=p, slot=p)
            assert L.tfr_fm_train_step(C.byref(t), p, 10, p, p, p, p, 30, p, p, p, p, sgd, p, 1 << 30, None) == -1, dim
            assert b"1 to 512" in L.tfr_last_error(), L.tfr_last_error()


@pytest.mark.skipif(not os.path.exists(NVCC), reason="needs the CUDA toolkit")
def test_fm_kernels_compile_for_every_case_without_spilling(tmp_path):
    """All 18 fm_forward_kernel instantiations and fm_err_kernel compile for sm_100a with no stack frame and no spills.
    CUDA 12.9: 32 registers for every UNITS = 1 case with VEC = 1 and for (4, 1, 1); 38 for the other UNITS = 1 cases with
    VEC = 4; (1, 32, 2) 32, (1, 32, 4) 40, (1, 32, 8) 39, (1, 32, 16) 64, (4, 32, 2) 48, (4, 32, 4) 66; fm_err_kernel 30."""
    from test_rank_users import _ptxas_lines
    obj, log = str(tmp_path / "fm.o"), str(tmp_path / "ptxas.txt")
    with open(log, "w") as f:
        subprocess.check_call([NVCC, "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-ccbin",
                               "/usr/bin/g++", "-Xcompiler", "-fPIC", "-Xptxas", "-v", "-c", FM_CU, "-o", obj],
                              stdout=f, stderr=subprocess.STDOUT)
    info = _ptxas_lines(log)
    want = {"void tfr::fm_forward_kernel<%d, %d, %d>" % c for c in fm_cases()} | {"tfr::fm_err_kernel"}
    assert want == set(info), sorted(want ^ set(info))
    for name, (regs, stack, st, ld) in info.items():
        assert (stack, st, ld) == (0, 0, 0), (name, info[name])


# ---- CPU: the oracle's FM at every dim ---------------------------------------------------------------------------------------
def _fp32_row_sums(indptr, indices, data, V):
    """s_f = sum_i fl(V_if x_i) and q_f = sum_i fl(t^2), each added in CSR order in fp32: the forward's own arithmetic,
    restated with numpy (one elementwise fp32 rounding per operation)."""
    n, d = len(indptr) - 1, V.shape[1]
    s, q = np.zeros((n, d), np.float32), np.zeros((n, d), np.float32)
    lens = np.diff(indptr)
    for k in range(int(lens.max(initial=0))):
        rows = np.flatnonzero(lens > k)
        p = indptr[rows] + k
        t = V[indices[p]] * data[p][:, None]
        s[rows] = s[rows] + t
        q[rows] = q[rows] + t * t
    return s, q


def _fp32_yhat(indptr, indices, data, w0, W, V):
    """The oracle's yhat restated with numpy: fl(fl(w0 + lin) + fl(0.5 * inter)), lin = sum_i fl(W_i x_i) in CSR order,
    inter = sum_f fl(fl(s_f^2) - q_f) in factor order, every sum in fp32."""
    s, q = _fp32_row_sums(indptr, indices, data, V)
    lens = np.diff(indptr)
    lin = np.zeros(len(lens), np.float32)
    for k in range(int(lens.max(initial=0))):
        rows = np.flatnonzero(lens > k)
        p = indptr[rows] + k
        lin[rows] = lin[rows] + W[indices[p]] * data[p]
    a = s * s - q
    inter = np.zeros(len(lens), np.float32)
    for f in range(V.shape[1]):
        inter = inter + a[:, f]
    return (w0[0] + lin) + np.float32(0.5) * inter


def _dense(indptr, indices, data, F):
    return sp.csr_matrix((data.astype(np.float64), indices, indptr), shape=(len(indptr) - 1, F)).toarray()


def _fm_tables(rng, F, d, scale=0.3):
    return (np.array([0.1], np.float32), rng.normal(0, scale, F).astype(np.float32),
            rng.normal(0, scale, (F, d)).astype(np.float32))


@pytest.mark.parametrize("d", ORACLE_DIMS)
def test_oracle_fm_forward_within_float64_bound(d):
    """The oracle's yhat and sums against forward.py:21-22 in float64 (np_oracle.fm_forward_dense), row by row, within
    the fp32 error bound of its sequential sums: with k non-zeros in the row, S_f = sum_i |V_if x_i| and
    Q_f = sum_i (V_if x_i)^2, |sums_f - exact| <= 2u (k + 1) S_f and
    |yhat - exact| <= 2u (k + d + 4) (|w0| + sum_i |W_i x_i| + sum_f (S_f^2 + Q_f)).  Its sums and yhat also equal, bit for
    bit, the same fp32 operations restated with numpy."""
    rng = np.random.default_rng(d)
    F, n = 60, 200
    indptr, indices, data = _fm_problem(rng, F, d, n, max_nnz=8, min_nnz=0)
    w0, W, V = _fm_tables(rng, F, d)
    y, sums = oracle.fm_forward(indptr, indices, data, w0, W, V, return_sums=True)
    X = _dense(indptr, indices, data, F)
    Vd = V.astype(np.float64)
    k = np.diff(indptr)
    S = np.abs(X) @ np.abs(Vd)
    err_s = np.abs(sums - X @ Vd)
    assert np.all(err_s <= 2 * U24 * (k + 1)[:, None] * S), "d=%d: sums off by up to %.3g" % (d, err_s.max())
    mass = abs(float(w0[0])) + np.abs(X) @ np.abs(W.astype(np.float64)) + (S * S + (X * X) @ (Vd * Vd)).sum(1)
    err_y = np.abs(y - np_oracle.fm_forward_dense(X, float(w0[0]), W, V))
    bound = 2 * U24 * (k + d + 4) * mass
    assert np.all(err_y <= bound), "d=%d: yhat off by %.3g (bound %.3g)" % (d, err_y.max(), bound[np.argmax(err_y)])
    s32, _ = _fp32_row_sums(indptr, indices, data, V)
    assert np.array_equal(sums.view(np.int32), s32.view(np.int32))
    assert np.array_equal(y.view(np.int32), _fp32_yhat(indptr, indices, data, w0, W, V).view(np.int32))


@pytest.mark.parametrize("flags", ORACLE_SGD_FLAGS)
def test_oracle_fm_sgd_step_matches_torch_autograd_at_dim_300(flags):
    _oracle_sgd_step_vs_autograd(flags, 300)


# ---- GPU: the forward at every sweep dim ------------------------------------------------------------------------------------
FWD_F, FWD_ROWS = 300, 517   # an odd row count: the last warp of every L < 32 geometry is partly filled


def _forward_rows(rng, F, n, binary):
    """Rows of 0, 1, 2, 3, 5, 8 and about 64 distinct features, x = 1 or uniform in [-2, 2)."""
    lens = rng.choice([0, 1, 2, 3, 5, 8, 64], n)
    lens = np.where(lens == 64, rng.integers(60, 69, n), lens)
    indptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    indices = np.concatenate([rng.choice(F, k, replace=False) for k in lens]).astype(np.int32)
    data = np.ones(len(indices), np.float32) if binary else rng.uniform(-2, 2, len(indices)).astype(np.float32)
    return indptr, indices, data


def _device_forward(indptr, indices, data, w0, W, V):
    import torch
    L = _lib.load()
    dev = torch.device("cuda")
    t = [torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in (indptr, indices, data, w0, W, V)]
    n, d = len(indptr) - 1, V.shape[1]
    yhat = torch.full((n,), float("nan"), device=dev)
    sums = torch.full((n, d), float("nan"), device=dev)
    _lib.check(L.tfr_fm_forward(n, *(a.data_ptr() for a in t), d, yhat.data_ptr(), sums.data_ptr(),
                                torch.cuda.current_stream().cuda_stream))
    return yhat.cpu().numpy(), sums.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("binary", [True, False], ids=["x01", "xreal"])
@pytest.mark.parametrize("d", FM_DIMS)
def test_fm_forward_every_dim_vs_oracle(d, binary):
    """sums bit for bit: the kernel and the oracle add fl(V_if x_i) and its square per factor in CSR order, one fp32
    rounding per operation (mul_rn / add_rn; the oracle is built with -ffp-contract=off).  yhat: both add the same
    a_f = fl(s_f^2 - q_f), the oracle one after the other and the kernel per lane and then across the lane group, to the
    same fl(w0 + lin); two fp32 sums of d terms differ by at most 2 (d - 1) u sum_f |a_f|, halved by the 0.5, plus the
    last addition's rounding on each side."""
    rng = np.random.default_rng(d + 1000 * binary)
    indptr, indices, data = _forward_rows(rng, FWD_F, FWD_ROWS, binary)
    w0, W, V = _fm_tables(rng, FWD_F, d, scale=0.1)
    y, sums = _device_forward(indptr, indices, data, w0, W, V)
    ref_y, ref_sums = oracle.fm_forward(indptr, indices, data, w0, W, V, return_sums=True)
    assert np.array_equal(sums.view(np.int32), ref_sums.view(np.int32)), \
        "d=%d: sums differ in %d entries" % (d, int((sums.view(np.int32) != ref_sums.view(np.int32)).sum()))
    s, q = _fp32_row_sums(indptr, indices, data, V)
    a = np.abs((s * s - q).astype(np.float64)).sum(1)
    bound = d * U24 * a + 4 * U24 * np.abs(ref_y)
    err = np.abs(y.astype(np.float64) - ref_y)
    assert np.all(err <= bound), "d=%d: yhat off by %.3g (bound %.3g)" % (d, err.max(), bound[np.argmax(err)])
    empty = np.diff(indptr) == 0
    assert empty.any() and np.all(y[empty] == w0[0])


# ---- GPU: the train step at every sweep dim against the oracle ----------------------------------------------------------------
F_SWEEP = 300


def _sweep_batches(rng, F):
    """A Zipf batch whose runs cross tiles, a batch of one row with one non-zero, and a batch whose ~400 rows all hold
    one hot feature (a run of hundreds of tiles: the fix-up's long-chain path)."""
    zipf = _fm_problem(rng, F, 0, 1500, 6, real_valued=True)
    one = (np.array([0, 1], np.int64), np.array([rng.integers(F)], np.int32), np.array([1.5], np.float32))
    hot = int(rng.integers(F))
    rest = np.delete(np.arange(F), hot)
    lens = rng.integers(1, 4, 400)
    indices = np.concatenate([np.r_[hot, rng.choice(rest, k - 1, replace=False)] for k in lens]).astype(np.int32)
    hot_batch = (np.concatenate([[0], np.cumsum(lens)]).astype(np.int64), indices, np.ones(len(indices), np.float32))
    return [zipf, one, hot_batch]


def _err_mass(yhat_ref, y, flags):
    x = yhat_ref.astype(np.float64)
    e = (1.0 / (1.0 + np.exp(-x)) if flags & _lib.LOSS_SIGMOID_CE else x) - y
    return float(np.abs(e).sum())


def _assert_fm_state(eng, orc, lr, e_mass, what):
    """test_fm_train_step_parity_adam's bar for W, V and their slots.  w0's gradient is one sum over the batch, sum_r e_r,
    which cancels under sigmoid-CE: w0 and its slots are judged against the mass of their terms, e_mass = sum |e_r| over
    the steps so far (lr * e_mass for w0, (1 - beta1) e_mass for m, 2 (1 - beta2) e_mass^2 for v)."""
    got = eng.get_tables()
    scale = {"w0": lr * e_mass, "m_w0": 0.1 * e_mass, "v_w0": 2e-3 * e_mass ** 2}
    for name in ("W", "V"):
        _assert_close(got[name], getattr(orc, name), "%s %s" % (what, name), max_abs=4 * lr + 1e-6)
        if not eng.sgd:
            for s in ("m_", "v_"):
                _assert_close(got[s + name], orc.slots[s + name], "%s %s%s" % (what, s, name))
    for name in ("w0",) + (() if eng.sgd else ("m_w0", "v_w0")):
        ref = float((orc.w0 if name == "w0" else orc.slots[name])[0])
        err = abs(float(got[name][0]) - ref)
        assert err <= RTOL * abs(ref) + RTOL * scale[name], "%s %s: |error| %.3g" % (what, name, err)


# Adam's first step on an entry is lr * g / (|g| + eps / sqrt(1 - beta2)): with eps = 1e-8 it is a sign function of
# a gradient that cancels to within fp32 noise of zero (d = 31 of the knob sweep: one V entry sums to 4e-7 from terms
# of total mass 0.64, and a few ulps of that mass move its update by 3e-4).  eps = 1e-3 bounds the update's sensitivity
# to lr / 0.03 per unit of gradient, so the bar measures the kernels' arithmetic rather than that conditioning; the
# slots, which hold the gradient sums themselves, are compared at the same bar.
ADAM_EPS = 1e-3


def _run_fm_vs_oracle(d, flags, seed, what):
    rng = np.random.default_rng(seed)
    lr = 1e-3 if flags & _lib.OPT_SGD else 1e-2
    eng, orc = _fm_pair(F_SWEEP, d, lr, 0.01, flags, seed=seed, eps=ADAM_EPS)
    e_mass = 0.0
    for s, (indptr, indices, data) in enumerate(_sweep_batches(rng, F_SWEEP)):
        y = rng.integers(0, 2, len(indptr) - 1).astype(np.float32)
        yhat = eng.train_step((indptr, indices, data), y).cpu().numpy()
        ref = orc.train_step(indptr, indices, data, y)
        _assert_close(yhat, ref, "%s step %d yhat" % (what, s))
        e_mass += _err_mass(ref, y, flags)
        _assert_fm_state(eng, orc, lr, e_mass, "%s step %d" % (what, s))
    assert eng.global_step == 3 == orc.s.global_step
    assert int((((eng.slot >> 32) & 0xffffffff) == 3).sum()) == 0   # no slot entry carries the next step's stamp


@pytest.mark.gpu
@pytest.mark.parametrize("d", FM_DIMS)
@pytest.mark.parametrize("model", list(FM_MODELS))
def test_fm_train_step_every_dim_vs_oracle(d, model):
    _run_fm_vs_oracle(d, FM_MODELS[model], d, "d=%d %s" % (d, model))


@pytest.mark.gpu
@pytest.mark.parametrize("d", KNOB_DIMS)
@pytest.mark.parametrize("max_units", SEG_UNITS)
@pytest.mark.parametrize("tile", SEG_TILES)
def test_fm_seg_tile_and_units_keep_oracle_parity(d, max_units, tile):
    with tuned(SEG_TILE=tile, SEG_MAX_UNITS=max_units):
        _run_fm_vs_oracle(d, 0, 2000 + d, "d=%d tile=%d units=%d" % (d, tile, max_units))


# ---- GPU: knobs that change launch geometry only keep every bit ---------------------------------------------------------------
FM_BIT_SHAPES = {"d15": (3000, 15), "d64": (3000, 64), "d260": (40000, 260)}   # (features, dim)
FM_BIT_STEPS = 3
_FM_BIT_BATCHES, _FM_BIT_REF = {}, {}


def _fm_bit_run(shape):
    F, d = FM_BIT_SHAPES[shape]
    if shape not in _FM_BIT_BATCHES:
        rng = np.random.default_rng(d)
        _FM_BIT_BATCHES[shape] = [(_fm_problem(rng, F, d, 2000, 6), rng.integers(0, 2, 2000).astype(np.float32))
                                  for _ in range(FM_BIT_STEPS)]
    eng, _ = _fm_pair(F, d, 1e-2, 0.01, 0, seed=d)
    outs = [eng.train_step(b, y).cpu().numpy() for b, y in _FM_BIT_BATCHES[shape]]
    return outs, eng.get_tables(), eng.opt_scalars()


@pytest.mark.gpu
@pytest.mark.parametrize("settings", BIT_SETTINGS, ids=lambda s: ",".join("%s=%d" % kv for kv in s.items()))
@pytest.mark.parametrize("shape", list(FM_BIT_SHAPES))
def test_fm_geometry_knobs_keep_every_bit(shape, settings):
    if shape not in _FM_BIT_REF:
        _FM_BIT_REF[shape] = _fm_bit_run(shape)
    with tuned(**settings):
        got = _fm_bit_run(shape)
    (oa, ta, sa), (ob, tb, sb) = _FM_BIT_REF[shape], got
    for s, (ya, yb) in enumerate(zip(oa, ob)):
        assert np.array_equal(ya.view(np.int32), yb.view(np.int32)), "%s yhat step %d" % (settings, s)
    assert set(ta) == set(tb)
    for n in ta:
        assert np.array_equal(ta[n].view(np.int32), tb[n].view(np.int32)), "%s %s" % (settings, n)
    for f in ("global_step", "beta1_power", "beta2_power", "lr_t", "g_mu", "se_sum"):
        assert getattr(sa, f) == getattr(sb, f), "%s %s" % (settings, f)


# ---- GPU: a batch of more than 1024 x 256 rows --------------------------------------------------------------------------------
@pytest.mark.gpu
def test_fm_large_batch_vs_oracle():
    """300000 rows: fm_err_kernel's grid is capped at TFR_MAX_PARTIALS CTAs and grid-strides, and w0's partial count is
    the cap.  Rows of 1 to 4 features, one from each quarter of the feature range, uniform inside it: a feature occurs
    about 6 times a batch.  (Zipf ids would give runs of ~10^5 cancelling terms, whose fp32 sums, the oracle's one after
    the other, differ from the exact ones by more than the 1e-5 bar.)"""
    F, d, n, lr, flags = 200000, 5, 300000, 1e-2, _lib.LOSS_SIGMOID_CE
    assert n > _lib.MAX_PARTIALS * 256
    rng = np.random.default_rng(7)
    eng, orc = _fm_pair(F, d, lr, 0.01, flags, seed=7, eps=ADAM_EPS)
    e_mass = 0.0
    for step in range(2):
        lens = rng.integers(1, 5, n)
        indptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
        nnz = int(indptr[-1])
        quarter = np.arange(nnz) - np.repeat(indptr[:-1], lens)
        indices = (quarter * (F // 4) + rng.integers(0, F // 4, nnz)).astype(np.int32)
        data = rng.uniform(0.5, 2.0, nnz).astype(np.float32)
        y = rng.integers(0, 2, n).astype(np.float32)
        yhat = eng.train_step((indptr, indices, data), y).cpu().numpy()
        ref = orc.train_step(indptr, indices, data, y)
        _assert_close(yhat, ref, "step %d yhat" % step)
        e_mass += _err_mass(ref, y, flags)
        _assert_fm_state(eng, orc, lr, e_mass, "step %d" % step)
    assert eng.global_step == 2


# ---- GPU: captured epochs and the driver at the new dims ------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("d", [65, 260])
def test_fm_graph_epoch_equals_eager_epoch(d):
    """run_epoch with captured graphs (each batch sorted once, then TFR_FM_PRESORTED) == the same steps launched eagerly,
    bit for bit."""
    from tf_recomm_b200.fm_engine import FmEngine
    rng = np.random.default_rng(d)
    F = 800
    chunks = [(_fm_problem(rng, F, d, 300, 6, real_valued=k % 2 == 1), rng.integers(0, 2, 300).astype(np.float32))
              for k in range(6)]
    engs = [FmEngine(F, d, 1e-2, 3e-2, flags=_lib.LOSS_SIGMOID_CE, seed=1) for _ in range(2)]
    for e, eng in enumerate(engs):
        batches = [eng.upload_csr(c, y) for c, y in chunks]
        for _ in range(3):
            eng.run_epoch(batches, use_graph=(e == 0))
    a, b = engs[0].get_tables(), engs[1].get_tables()
    assert set(a) == set(b)
    for k in a:
        assert np.array_equal(a[k].view(np.int32), b[k].view(np.int32)), k
    assert engs[0].global_step == engs[1].global_step == 3 * 6


@pytest.mark.gpu
def test_fm_driver_at_dim_65(tmp_path):
    """`python fm.py --dataset syn --d 65 --users --items --skills --iter 3 --synthetic 2000`."""
    import json
    import fm as fm_driver
    res = fm_driver.main(["--dataset", "syn", "--d", "65", "--users", "--items", "--skills", "--iter", "3", "--synthetic",
                          "2000", "--data_folder", str(tmp_path), "--seed", "0", "--folds", "2", "--batch", "500"])
    folder = os.path.join(str(tmp_path), "syn", "uis65")
    for run in ("0", "1"):
        r = json.load(open(os.path.join(folder, run, "results.json")))
        assert set(r["metrics"]) == {"ACC", "AUC", "NLL"}
        assert np.load(os.path.join(folder, run, "vectors-65.npy")).shape[-1] == 65
    assert len(res) == 2 and all(np.isfinite(r["NLL"]) for r in res), res
