"""The float64 row solver of csrc/fold_in.cuh (Gram of a row's ratings in shared memory, Cholesky, substitution) at every
dim it takes, every tile and chunk edge, and in every consumer: tfr_fold_in_users (FiRatings), the ALS half-sweeps
(FiRatings, light rows and split heavy rows), the iALS half-sweeps and fold_in_implicit (FiImplicit, started from G) and
tfr_gram_rows (FiPlain's tile Gram).  Every solved row is compared with np.linalg.solve on the same float64 system.

The solver's geometry depends on D = dim + 1 (with the bias column) or dim: the staged tile is [FI_TILE][Dp] doubles,
Dp = ceil(D / 4) * 4; each thread owns 4 x 4 blocks of the packed triangle, a second one once there are more than
FI_THREADS blocks (D >= 89); the solving warp holds entry i in register v[i / 32], so D = 32 / 33, 64 / 65, 96 / 97 and
128 / 129 are register boundaries.  Heavy rows (more than ALS_CHUNK ratings) are split into chunks whose float64 partials
are summed in chunk order.  The GPU tests run every dim 1..128 with rows of every length class around those edges; the
CPU tests mirror the shared-memory layout, check that the sweeps reach every class, and pin a bit-exact numpy model of
tfr_gram_rows.  The failure tests run the guarded paths the kernels document: a partner id just outside the fixed side's
range makes the row keep its previous values, counts it in *n_failed, and poisons both objectives.
"""
import os
import re

import numpy as np
import pytest
import torch

from test_als import ALS_FLAGS, loss as svd_loss, residuals
from test_als import half_ref as als_half_ref
from test_fold_in import FLAG_SETS, _c_fold, _rows, fold_ref
from test_fold_in import _engine as fold_engine
from test_ials import _Chunk, dense_loss, gram_loss, merge
from test_ials import half_ref as ials_half_ref
from tf_recomm_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "tf-recomm_b200", "csrc")
NEEDS_CUDA = pytest.mark.skipif(not torch.cuda.is_available(), reason="needs a CUDA device")


def _constant(src, name):
    with open(os.path.join(CSRC, src)) as f:
        m = re.search(r"constexpr int [^;]*\b%s = (\d+)" % name, f.read())
    assert m, (src, name)
    return int(m.group(1))


FI_TILE = _constant("fold_in.cuh", "FI_TILE")
FI_THREADS = _constant("fold_in.cuh", "FI_THREADS")
FI_MAX_DIM = _constant("fold_in.cuh", "FI_MAX_DIM")
GRAM_ROWS = _constant("ials.cu", "GRAM_ROWS")

SMEM_BLOCK, SMEM_SM, SMEM_RESERVED = 227 * 1024, 228 * 1024, 1024   # sm_100: per block, per SM, reserved per block
STATIC_SMEM = 16   # each solver kernel's static __shared__ (s_bad, one int), rounded up

DIMS = list(range(1, FI_MAX_DIM + 1))
FORMS = {"ratings": (1, False), "implicit": (0, True), "plain": (0, False)}   # FiForm: (extra rows, weighted)
CHUNK = 64                                      # ALS_CHUNK of the sweeps: two staging tiles
KNOB_DIMS = [31, 32, 33, 64, 65, 127, 128]      # each side of the register boundaries
KNOBS = [(1, 32), (33, 64), (4096, 4096), (1 << 20, 1 << 20)]   # ALS_CHUNK -> tfr_als_chunk()
FAIL_DIMS = [1, 33, 128]
GRAM_NS = [0, 1, 31, 32, 33, 1023, 1024, 1025, 3 * 1024 + 17]
REG, LAM = 0.05, float(np.float32(0.05))


# ---- the geometry, mirrored from fold_in.cuh ----------------------------------------------------------------------------
def _align16(x):
    return (x + 15) & ~15


def _tri(i, j=0):
    return i * (i + 1) // 2 + j


def fi_smem(dim, form):
    """fi_smem<F>(dim): byte offsets (tri, rhs, x, y, w, item, total) of one CTA's dynamic shared memory."""
    extra, weighted = FORMS[form]
    D = dim + extra
    Dp = (D + 3) // 4 * 4
    tri = 0
    rhs = _align16(_tri(D) * 8)
    x = _align16(rhs + D * 8)
    y = x + FI_TILE * Dp * 8
    w = y + FI_TILE * 8
    item = w + (FI_TILE * 8 if weighted else 0)
    return dict(tri=tri, rhs=rhs, x=x, y=y, w=w, item=item, total=item + FI_TILE * 4)


def geometry(dim, form):
    """(D, Dp, n_blk, solve registers in use) of a row system of `form` at `dim`."""
    D = dim + FORMS[form][0]
    Dp = (D + 3) // 4 * 4
    Db = Dp // 4
    return D, Dp, Db * (Db + 1) // 2, (D + 31) // 32


def fold_counts(d):
    """Fold-in rows: 1, 2, the tile edges, d - 1, d, d + 1 and about 3000 ratings (d - 1 = 0 at d = 1: an empty row)."""
    return [1, 2, FI_TILE - 1, FI_TILE, FI_TILE + 1, d - 1, d, d + 1, 3001]


def row_classes():
    """Row lengths around the tile and chunk edges (CHUNK = 2 tiles): empty, one, a tile -1 / exact / +1, a chunk exactly, a
    heavy row whose last chunk is 1, two full chunks, two chunks + 1, and a row of four chunks."""
    return [0, 1, FI_TILE - 1, FI_TILE, FI_TILE + 1, CHUNK, CHUNK + 1, 2 * CHUNK, 2 * CHUNK + 1, 3 * CHUNK + 8]


def class_counts(d):
    return row_classes() + [max(d - 1, 0), d, d + 1]


# ---- problems --------------------------------------------------------------------------------------------------------------
ALS_U, ALS_I = 200, 150
IALS_U, IALS_I = 260, 260


def als_problem(d, seed):
    """Explicit ratings: user k and item k (k < number of classes) have class_counts(d)[k] ratings each, from filler
    partners (ids >= the number of classes), the last one a duplicate of the first; the fillers also rate each other."""
    rng = np.random.default_rng(seed)
    counts = class_counts(d)
    nc = len(counts)
    us, its = [], []
    for k, c in enumerate(counts):
        f, g = rng.integers(nc, ALS_I, c), rng.integers(nc, ALS_U, c)
        if c >= 2:
            f[-1], g[-1] = f[0], g[0]
        us += [np.full(c, k), g]
        its += [f, np.full(c, k)]
    us.append(rng.integers(nc, ALS_U, 6000))
    its.append(rng.integers(nc, ALS_I, 6000))
    users, items = np.concatenate(us), np.concatenate(its)
    perm = rng.permutation(len(users))
    rates = rng.integers(1, 6, len(users)).astype(np.float32)
    return users[perm].astype(np.int32), items[perm].astype(np.int32), rates


def ials_problem(d, seed):
    """Implicit feedback: user k and item k have class_counts(d)[k] distinct filler partners, plus one duplicate entry (merged
    away), weights in quarters so that merged sums are exact; the fillers interact among themselves."""
    rng = np.random.default_rng(seed)
    counts = class_counts(d)
    nc = len(counts)
    us, its = [], []
    for k, c in enumerate(counts):
        f, g = rng.choice(np.arange(nc, IALS_I), c, replace=False), rng.choice(np.arange(nc, IALS_U), c, replace=False)
        if c >= 1:
            f, g = np.append(f, f[0]), np.append(g, g[0])
        us += [np.full(len(f), k), g]
        its += [f, np.full(len(g), k)]
    us.append(rng.integers(nc, IALS_U, 6000))
    its.append(rng.integers(nc, IALS_I, 6000))
    users, items = np.concatenate(us), np.concatenate(its)
    perm = rng.permutation(len(users))
    w = (rng.integers(1, 9, len(users)) / 4.0).astype(np.float32)
    return users[perm].astype(np.int32), items[perm].astype(np.int32), w


KNOB_U, KNOB_I = 40, 4400


def knob_counts():
    """User rows of the chunk-knob problem: light under every knob up to heavy under every knob but 2^20."""
    return [0, 1, 31, 32, 33, 64, 65, 96, 129, 200, 4097]


def knob_problem(seed, heavy_fillers):
    """Users k < len(knob_counts()) rate knob_counts()[k] distinct items (weights in quarters), in an order that does not
    depend on the rest; filler users rate 20 items each, or 300 with heavy_fillers (heavy under chunks 32 and 64).  The
    controlled entries come first in one problem and last in the other, so each controlled row has the same CSR row (and
    the same merged weights) in both."""
    rng = np.random.default_rng(1234)
    counts = knob_counts()
    nc = len(counts)
    cu = np.concatenate([np.full(c, k) for k, c in enumerate(counts)])
    ci = np.concatenate([rng.choice(KNOB_I, c, replace=False) for c in counts])
    cw = rng.integers(1, 9, len(cu)) / 4.0
    cr = rng.integers(1, 6, len(cu))
    frng = np.random.default_rng(seed)
    per = 300 if heavy_fillers else 20
    fu = np.repeat(np.arange(nc, KNOB_U), per)
    fi = frng.integers(0, KNOB_I, len(fu))
    fw, fr = frng.integers(1, 9, len(fu)) / 4.0, frng.integers(1, 6, len(fu))
    parts = [(cu, ci, cw, cr), (fu, fi, fw, fr)]
    if heavy_fillers:
        parts.reverse()
    u, i, w, r = (np.concatenate(x) for x in zip(*parts))
    return u.astype(np.int32), i.astype(np.int32), w.astype(np.float32), r.astype(np.float32)


# ---- the bit-exact model of tfr_gram_rows --------------------------------------------------------------------------------------
def _packed(d):
    ia, ib = np.tril_indices(d)
    order = np.lexsort((ib, ia))   # packed row-major lower triangle
    return ia[order], ib[order]


def gram_model(X):
    """tfr_gram_rows's bits: CTA b sums entry (a, b) of rows [b GRAM_ROWS, (b + 1) GRAM_ROWS) in row order from 0.0 as
    fma(x_a, x_b, acc); gram_combine_kernel sums the partials in CTA order from 0.0.  The rows are fp32, so x_a x_b is exact
    in float64 and fma(x_a, x_b, acc) == acc + x_a x_b."""
    X = np.asarray(X, np.float32).astype(np.float64)
    ia, ib = _packed(X.shape[1])
    G = np.zeros(len(ia))
    for b0 in range(0, len(X), GRAM_ROWS):
        acc = np.zeros(len(ia))
        for x in X[b0:b0 + GRAM_ROWS]:
            acc = acc + x[ia] * x[ib]
        G = G + acc
    return G


def _bar(got, ref):
    """Rows of got (float64 of the fp32 results) outside fold-in's bar 2^-24 |ref| + 1e-10 max|ref| (per row)."""
    tol = 2.0 ** -24 * np.abs(ref) + 1e-10 * np.abs(ref).max(axis=1, keepdims=True)
    return np.nonzero((np.abs(got - ref) > tol).any(axis=1))[0]


def _assert_bar(got, ref, what):
    bad = _bar(np.asarray(got, np.float64), ref)
    assert len(bad) == 0, (what, bad[:10].tolist(), float(np.abs(got - ref)[bad].max()))


def _u32(a):
    return np.ascontiguousarray(a).view(np.uint32)


# ---- CPU -------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("form", sorted(FORMS))
def test_shared_memory_layout_at_every_dim(form):
    """For every dim 1..FI_MAX_DIM: the staged tile x (read as double2) is 16-byte aligned, every other array 8-byte
    aligned, and two CTAs' dynamic + static shared memory fit an SM, as __launch_bounds__(FI_THREADS, 2) assumes."""
    for dim in DIMS:
        s = fi_smem(dim, form)
        D, Dp, _, _ = geometry(dim, form)
        assert s["x"] % 16 == 0, (form, dim, s)
        assert all(s[k] % 8 == 0 for k in ("rhs", "y", "w")) and s["item"] % 4 == 0, (form, dim, s)
        assert s["rhs"] >= _tri(D) * 8 and s["x"] >= s["rhs"] + D * 8, (form, dim, s)   # nothing overlaps
        block = s["total"] + STATIC_SMEM
        assert block <= SMEM_BLOCK and 2 * (block + SMEM_RESERVED) <= SMEM_SM, (form, dim, block)


def test_the_sweeps_reach_every_geometry_class():
    """The dims the GPU tests sweep reach, per form: every Dp, every number of solve registers in use and the D one past
    each register boundary, and both sides of n_blk > FI_THREADS; the knob dims sit on both sides of three boundaries."""
    n_regs = (FI_MAX_DIM + 1 + 31) // 32
    for form, consumers in (("ratings", "fold-in, ALS"), ("implicit", "iALS"), ("plain", "Gram")):
        geo = [geometry(d, form) for d in DIMS]
        Ds = {g[0] for g in geo}
        D_max = FI_MAX_DIM + FORMS[form][0]
        assert {g[1] for g in geo} == set(range(4, (D_max + 3) // 4 * 4 + 1, 4)), consumers
        assert {g[3] for g in geo} == set(range(1, (D_max + 31) // 32 + 1)), consumers
        assert {32 * k + 1 for k in range(1, n_regs) if 32 * k + 1 <= D_max} <= Ds, consumers
        assert any(g[2] > FI_THREADS for g in geo) and any(g[2] <= FI_THREADS for g in geo), consumers
    for b in (32, 64, 128):
        assert {b - 1, b, b + 1} & set(KNOB_DIMS) and any(d < b for d in KNOB_DIMS) and any(d >= b for d in KNOB_DIMS)


@pytest.mark.parametrize("d", [1, 2, 33, 64, 128])
def test_the_problems_reach_every_row_length_class(d):
    """Both sides of the ALS and iALS problems have rows of every class of row_classes() (iALS after merging), fold-in
    rows cover the tile edges, and the knob problem has rows light and heavy under each knob value."""
    want = set(row_classes())
    assert {0, 1, FI_TILE - 1, FI_TILE, FI_TILE + 1, CHUNK, CHUNK + 1, 2 * CHUNK, 2 * CHUNK + 1} <= want
    assert max(want) > 3 * CHUNK
    users, items, _ = als_problem(d, seed=d)
    for ids, n in ((users, ALS_U), (items, ALS_I)):
        assert want <= set(np.bincount(ids, minlength=n).tolist())
    users, items, w = ials_problem(d, seed=d)
    mu_, mi_, _ = merge(users, items, w)
    for ids, n in ((mu_, IALS_U), (mi_, IALS_I)):
        assert want <= set(np.bincount(ids, minlength=n).tolist())
    assert {FI_TILE - 1, FI_TILE, FI_TILE + 1, d} <= set(fold_counts(d)) and max(fold_counts(d)) > 3000
    counts = knob_counts()
    for _, chunk in KNOBS:
        assert any(0 < c <= chunk for c in counts) and (chunk == 1 << 20 or any(c > chunk for c in counts))
        assert chunk >= 1 << 20 or any(c % chunk == 1 and c > chunk for c in counts)   # a last chunk of one
    for heavy in (False, True):
        u, i, w, r = knob_problem(5, heavy)
        assert np.array_equal(np.bincount(merge(u, i, w)[0], minlength=KNOB_U)[:len(counts)], counts)
        assert np.array_equal(np.bincount(u, minlength=KNOB_U)[:len(counts)], counts)


def test_the_knob_values_give_the_chunks_the_tests_expect():
    L = _lib.load()
    old = _lib.tune_get("ALS_CHUNK")
    try:
        for knob, chunk in KNOBS + [(CHUNK, CHUNK)]:
            _lib.tune_set("ALS_CHUNK", knob)
            assert L.tfr_als_chunk() == chunk
    finally:
        _lib.tune_set("ALS_CHUNK", old)


@pytest.mark.parametrize("d", [1, 5, 31, 64, 97, 128])
def test_gram_model_is_the_float64_gram(d):
    """The bit model of tfr_gram_rows meets the 1e-12 |X|^T |X| bar against X^T X, across CTA edges, and its first CTA's
    sum is numpy's own sequential (cumulative) sum of the products: the model is a plain in-order sum."""
    rng = np.random.default_rng(d)
    ia, ib = _packed(d)
    for n in (0, 1, 33, GRAM_ROWS, GRAM_ROWS + 1, 2 * GRAM_ROWS + 17):
        X = rng.normal(0, 0.5, (n, d)).astype(np.float32)
        got = gram_model(X)
        Xd = X.astype(np.float64)
        ref, bound = (Xd.T @ Xd)[ia, ib], (np.abs(Xd).T @ np.abs(Xd))[ia, ib]
        assert (np.abs(got - ref) <= 1e-12 * bound).all(), (d, n)
        if 0 < n <= GRAM_ROWS:
            seq = np.cumsum(Xd[:, ia] * Xd[:, ib], axis=0)[-1]
            assert np.array_equal(got.view(np.uint64), seq.view(np.uint64)), (d, n)
    assert not gram_model(np.zeros((0, d), np.float32)).any()


# ---- GPU: helpers --------------------------------------------------------------------------------------------------------------
def _gram_rows(L, F, n, d, stride):
    out = torch.empty(d * (d + 1) // 2, dtype=torch.float64, device="cuda")
    nbytes = _lib.check(L.tfr_gram_workspace_bytes(n, d))
    ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    _lib.check(L.tfr_gram_rows(F.data_ptr() if n else 0, n, d, stride, out.data_ptr(), ws.data_ptr(), nbytes,
                               torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return out.cpu().numpy()


def _svd_engine(U, I, d, flags, seed=5):
    from tf_recomm_b200 import init
    from tf_recomm_b200.engine import SvdEngine
    tabs = init.init_tables(U, I, d, seed=seed, bias_init="truncated_normal")
    tabs["user_feat"] *= 10
    tabs["item_feat"] *= 10
    tabs["mu"][:] = 3.5
    return SvdEngine(U, I, d, 1e-3, REG, flags=flags, tables=tabs)


TABLES = ("mu", "user_bias", "item_bias", "user_feat", "item_feat")


def _tables(eng):
    torch.cuda.synchronize()
    return {n: eng.t[n].cpu().numpy().copy() for n in TABLES}


def _restore(eng, T):
    for n, a in T.items():
        eng.t[n].copy_(torch.from_numpy(a.reshape(eng.t[n].shape)))


def _same(T, U_, names):
    return all(np.array_equal(_u32(T[n]), _u32(U_[n])) for n in names)


def _als_half(eng, data, side):
    T = eng.t
    with torch.cuda.device(eng.device):
        if side == "user":
            eng._half_sweep(data, REG, data.by_user, data.user_plan, (T["item_feat"], T["item_bias"], eng.I),
                            (T["user_feat"], T["user_bias"]))
        else:
            eng._half_sweep(data, REG, data.by_item, data.item_plan, (T["user_feat"], T["user_bias"], eng.U),
                            (T["item_feat"], T["item_bias"]))


def _ials_half(eng, data, side, alpha):
    T = eng.t
    with torch.cuda.device(eng.device):
        if side == "user":
            eng._gram(T["item_feat"], eng.I, data.item_gram, data.workspace)
            eng._ials_half(data, alpha, LAM, data.by_user, data.user_plan, (T["item_feat"], eng.I, data.item_gram),
                           (T["user_feat"], T["user_bias"]))
        else:
            eng._gram(T["user_feat"], eng.U, data.user_gram, data.workspace)
            eng._ials_half(data, alpha, LAM, data.by_item, data.item_plan, (T["user_feat"], eng.U, data.user_gram),
                           (T["item_feat"], T["item_bias"]))


def _als_ref(T, side, users, items, rates, flags):
    if side == "user":
        return als_half_ref(T["item_feat"], T["item_bias"], T["mu"][0], users, items, rates, len(T["user_bias"]), REG,
                            flags)
    return als_half_ref(T["user_feat"], T["user_bias"], T["mu"][0], items, users, rates, len(T["item_bias"]), REG, flags)


def _ials_ref(T, side, merged, alpha):
    mu_, mi_, mw_ = merged
    if side == "user":
        return ials_half_ref(T["item_feat"], mu_, mi_, mw_, len(T["user_feat"]), alpha, LAM)
    return ials_half_ref(T["user_feat"], mi_, mu_, mw_, len(T["item_feat"]), alpha, LAM)


def _with_bias(T, side):
    return np.hstack([T[side + "_feat"].astype(np.float64), T[side + "_bias"].astype(np.float64)[:, None]])


OTHER = {"user": "item", "item": "user"}


# ---- GPU: Gram ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("d", DIMS)
@pytest.mark.gpu
@NEEDS_CUDA
def test_gram_rows_bit_for_bit(d):
    """tfr_gram_rows equals gram_model bit for bit for row counts at the tile and CTA edges, on tables of stride dim,
    dim + 3 and 3 dim (the engine's interleaved [var|m|v] layout), the padding filled with other values."""
    L = _lib.load()
    rng = np.random.default_rng(1000 + d)
    for n in GRAM_NS:
        X = rng.normal(0, 0.5, (n, d)).astype(np.float32)
        want = gram_model(X)
        for stride in (d, d + 3, 3 * d):
            F = rng.normal(0, 4.0, (n, stride)).astype(np.float32)
            F[:, :d] = X
            got = _gram_rows(L, torch.from_numpy(F).cuda(), n, d, stride)
            assert np.array_equal(got.view(np.uint64), want.view(np.uint64)), (n, stride)


# ---- GPU: fold-in --------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("d", DIMS)
@pytest.mark.gpu
@NEEDS_CUDA
def test_fold_in_rows(d):
    """tfr_fold_in_users under the four flag sets and two regs, rows of 1, 2, 31, 32, 33, d - 1, d, d + 1 and 3001
    ratings with duplicates: every entry within 2^-24 |ref| + 1e-10 max|ref| of fold_ref, info 0."""
    I = 3000
    eng, tabs = fold_engine(40, I, d)
    counts = fold_counts(d)
    rows, items, rates = _rows(I, d, counts, seed=d)
    indptr, it, rt = eng._csr_by_user(rows, items, rates, n_rows=len(counts))
    for flags in FLAG_SETS:
        for reg in (0.05, 1e-3):
            feat, bias, info = (a.cpu().numpy() for a in _c_fold(eng, indptr, it, rt, reg, flags=flags))
            assert not info.any(), (flags, reg, info)
            got = np.hstack([feat.astype(np.float64), bias.astype(np.float64)[:, None]])
            ref = np.stack([fold_ref(tabs["item_feat"], tabs["item_bias"], tabs["mu"][0], items[rows == r],
                                     rates[rows == r], reg, flags) for r in range(len(counts))])
            _assert_bar(got, ref, (flags, reg))


# ---- GPU: ALS ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("d", DIMS)
@pytest.mark.gpu
@NEEDS_CUDA
def test_als_half_sweeps(d):
    """ALS at ALS_CHUNK = 64, flags {0, REG_BIAS}, Adam (interleaved tables) and SGD: each half-step within the bar of
    half_ref from the GPU's tables just before it, light and heavy rows of every class on both sides; the fixed side and mu
    unchanged bit for bit; the user half equals tfr_fold_in_users bit for bit on every light row; the objective's sums
    within 1e-12 of numpy's; the mu step is fl32(mu + mean e); no row fails."""
    users, items, rates = als_problem(d, seed=d)
    n_u, n_i = np.bincount(users, minlength=ALS_U), np.bincount(items, minlength=ALS_I)
    for flags in ALS_FLAGS:
        for sgd in (False, True):
            with _Chunk(CHUNK):
                eng = _svd_engine(ALS_U, ALS_I, d, flags | (_lib.OPT_SGD if sgd else 0), seed=d)
                data = eng.als_data(users, items, rates)
            assert data.chunk == CHUNK
            assert data.user_plan.heavy.numel() == (n_u > CHUNK).sum() >= 4
            assert data.item_plan.heavy.numel() == (n_i > CHUNK).sum() >= 4
            T0 = _tables(eng)
            folded = eng.fold_in(users, items, rates, n=ALS_U, reg=REG)
            _als_half(eng, data, "user")
            T1 = _tables(eng)
            _assert_bar(_with_bias(T1, "user"), _als_ref(T0, "user", users, items, rates, flags), (flags, sgd, "user"))
            assert _same(T0, T1, ("mu", "item_feat", "item_bias"))
            light = n_u <= CHUNK
            assert np.array_equal(_u32(folded.feat.cpu().numpy())[light], _u32(T1["user_feat"])[light])
            assert np.array_equal(_u32(folded.bias.cpu().numpy())[light], _u32(T1["user_bias"])[light])
            _als_half(eng, data, "item")
            T2 = _tables(eng)
            _assert_bar(_with_bias(T2, "item"), _als_ref(T1, "item", users, items, rates, flags), (flags, sgd, "item"))
            assert _same(T1, T2, ("mu", "user_feat", "user_bias"))
            # the objective: out6 = (L, sum e^2, sum e, sum n |x|^2, sum n b^2, N)
            obj = eng.training_objective(data, reg=REG)
            o = data.objective.cpu().numpy()
            e = residuals(T2, users, items, rates)
            f = {k: T2[k].astype(np.float64) for k in TABLES}
            pen = (f["user_feat"][users] ** 2).sum() + (f["item_feat"][items] ** 2).sum()
            pen_b = (f["user_bias"][users] ** 2).sum() + (f["item_bias"][items] ** 2).sum()
            want = svd_loss(T2, users, items, rates, REG, flags)
            assert abs(obj["loss"] - want) <= 1e-12 * want and obj["n"] == len(users) == o[5]
            assert abs(o[1] - e @ e) <= 1e-12 * (e @ e) and abs(o[2] - e.sum()) <= 1e-12 * np.abs(e).sum()
            assert abs(o[3] - pen) <= 1e-12 * pen and abs(o[4] - pen_b) <= 1e-12 * pen_b
            with torch.cuda.device(eng.device):
                eng._objective(data, REG, eng.t["mu"].data_ptr())
            T3 = _tables(eng)
            assert T3["mu"][0] == np.float32(T2["mu"][0] + e.mean())
            assert _same(T2, T3, TABLES[1:])
            assert int(data.failed.item()) == 0


# ---- GPU: iALS -----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("d", DIMS)
@pytest.mark.gpu
@NEEDS_CUDA
def test_ials_half_sweeps(d):
    """iALS at ALS_CHUNK = 64 for alpha 0, 1 and 40: each half-step within the bar of test_ials.half_ref, light and heavy
    rows of every class on both sides (after merging); solved rows' biases exactly 0; the fixed side unchanged bit for bit;
    the objective within 1e-12 of gram_loss and of the dense loss; fold_in_implicit equals the user half-sweep bit for bit
    with every row light.  Adam tables at even dims, SGD at odd ones."""
    users, items, w = ials_problem(d, seed=d)
    merged = merge(users, items, w)
    n_u = np.bincount(merged[0], minlength=IALS_U)
    n_i = np.bincount(merged[1], minlength=IALS_I)
    with _Chunk(CHUNK):
        eng = _svd_engine(IALS_U, IALS_I, d, _lib.OPT_SGD if d % 2 else 0, seed=d)
        data = eng.ials_data(users, items, w)
    assert data.chunk == CHUNK and data.by_user.partner.numel() == len(merged[0])
    assert data.user_plan.heavy.numel() == (n_u > CHUNK).sum() >= 4
    assert data.item_plan.heavy.numel() == (n_i > CHUNK).sum() >= 4
    for alpha in (0.0, 1.0, 40.0):
        T0 = _tables(eng)
        _ials_half(eng, data, "user", alpha)
        T1 = _tables(eng)
        _assert_bar(T1["user_feat"], _ials_ref(T0, "user", merged, alpha), (alpha, "user"))
        assert not T1["user_bias"].view(np.uint32).any()
        assert _same(T0, T1, ("mu", "item_feat", "item_bias"))
        _ials_half(eng, data, "item", alpha)
        T2 = _tables(eng)
        _assert_bar(T2["item_feat"], _ials_ref(T1, "item", merged, alpha), (alpha, "item"))
        assert not T2["item_bias"].view(np.uint32).any()
        assert _same(T1, T2, ("mu", "user_feat", "user_bias"))
        o = eng.implicit_objective(data, alpha, reg=REG)
        want = gram_loss(T2["user_feat"], T2["item_feat"], *merged, alpha, LAM)
        assert abs(o["loss"] - want) <= 1e-12 * want, (alpha, o, want)
        dense = dense_loss(T2["user_feat"], T2["item_feat"], *merged, alpha, LAM)
        assert abs(o["loss"] - dense) <= 1e-12 * dense and o["n"] == len(merged[0])
    assert int(data.failed.item()) == 0
    with _Chunk(1 << 20):
        whole = eng.ials_data(users, items, w)
    assert whole.user_plan.heavy.numel() == 0
    f = eng.fold_in_implicit(users, items, w, n=IALS_U, alpha=40.0, reg=REG)
    _ials_half(eng, whole, "user", 40.0)
    assert np.array_equal(_u32(f.feat.cpu().numpy()), _u32(eng.t["user_feat"].cpu().numpy()))
    assert not f.info.cpu().numpy().any() and int(whole.failed.item()) == 0


# ---- GPU: the chunk knob ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("d", KNOB_DIMS)
@pytest.mark.parametrize("solver", ["als", "ials"])
@pytest.mark.gpu
@NEEDS_CUDA
def test_chunk_knob(solver, d):
    """The user half-sweep under ALS_CHUNK 1, 33, 4096 and 2^20 (chunks 32, 64, 4096, 2^20), in two problems that share
    the controlled rows but not the rest (light fillers in one, fillers heavy under chunks 32 and 64 in the other): a row
    keeps its bits under every knob that leaves it light, whichever other rows are heavy; a heavy row meets the bar under
    every knob; a row split the same way in both problems has the same bits in both."""
    counts = knob_counts()
    nc = len(counts)
    eng = _svd_engine(KNOB_U, KNOB_I, d, _lib.REG_BIAS if solver == "als" else 0, seed=d)
    T0 = _tables(eng)
    results = {}
    for heavy_fillers in (False, True):
        u, i, w, r = knob_problem(d, heavy_fillers)
        if solver == "als":
            ref = _als_ref(T0, "user", u, i, r, _lib.REG_BIAS)
        else:
            merged = merge(u, i, w)
            ref = _ials_ref(T0, "user", merged, 40.0)
        n_u = np.bincount(u if solver == "als" else merged[0], minlength=KNOB_U)
        for knob, chunk in KNOBS:
            with _Chunk(knob):
                data = eng.als_data(u, i, r) if solver == "als" else eng.ials_data(u, i, w)
            assert data.chunk == chunk
            assert data.user_plan.heavy.numel() == (n_u > chunk).sum()
            _restore(eng, T0)
            if solver == "als":
                _als_half(eng, data, "user")
            else:
                _ials_half(eng, data, "user", 40.0)
            T = _tables(eng)
            got = _with_bias(T, "user") if solver == "als" else T["user_feat"].astype(np.float64)
            _assert_bar(got, ref, (heavy_fillers, chunk))
            assert int(data.failed.item()) == 0
            results[heavy_fillers, chunk] = np.hstack([_u32(T["user_feat"]), _u32(T["user_bias"])[:, None]])
    for r in range(nc):
        light = [results[h, c][r] for h in (False, True) for _, c in KNOBS if counts[r] <= c]
        assert all(np.array_equal(light[0], x) for x in light), r
        for _, c in KNOBS:
            assert np.array_equal(results[False, c][r], results[True, c][r]), (r, c)


# ---- GPU: failure paths --------------------------------------------------------------------------------------------------------
def _poison_sites(indptr, n_fixed):
    """(row, CSR position, bad id) in three places of the controlled rows: a light row of FI_TILE + 1 ratings, chunk 0 of
    the row of 3 CHUNK + 8, and the last chunk (of one rating) of the row of 2 CHUNK + 1."""
    cls = row_classes()
    sites = []
    for count, k, bad in ((FI_TILE + 1, 5, n_fixed), (3 * CHUNK + 8, 7, -1), (2 * CHUNK + 1, 2 * CHUNK, n_fixed)):
        r = cls.index(count)
        assert indptr[r + 1] - indptr[r] == count
        sites.append((r, int(indptr[r]) + k, bad))
    return sites


@pytest.mark.parametrize("d", FAIL_DIMS)
@pytest.mark.parametrize("solver", ["als", "ials"])
@pytest.mark.gpu
@NEEDS_CUDA
def test_out_of_range_partner_ids(solver, d):
    """One partner id set to n_fixed or -1 in a light row, in chunk 0 of a heavy row and in the last chunk of another heavy
    row (the guard of fi_gram: `it >= 0 && it < n_fixed`, never read through): the half-sweep counts 3 failed rows, those
    rows keep their previous bits (feature and bias), no NaN enters any table, and every other row has the bits of the same
    half-sweep without the poison.  The same poison in the user CSR makes the objective NaN (its guard poisons the sums)."""
    if solver == "als":
        users, items, vals = als_problem(d, seed=d)
        U, I = ALS_U, ALS_I
    else:
        users, items, vals = ials_problem(d, seed=d)
        U, I = IALS_U, IALS_I
    with _Chunk(CHUNK):
        eng = _svd_engine(U, I, d, _lib.REG_BIAS if solver == "als" else 0, seed=d)
        data = eng.als_data(users, items, vals) if solver == "als" else eng.ials_data(users, items, vals)
    T0 = _tables(eng)

    def half(side):
        _restore(eng, T0)
        data.failed.zero_()
        if solver == "als":
            _als_half(eng, data, side)
        else:
            _ials_half(eng, data, side, 40.0)
        return _tables(eng), int(data.failed.item())

    def objective():
        if solver == "als":
            return eng.training_objective(data, reg=REG)["loss"]
        return eng.implicit_objective(data, 40.0, reg=REG)["loss"]

    for side in ("user", "item"):
        csr = data.by_user if side == "user" else data.by_item
        n_fixed = I if side == "user" else U
        clean_ids = csr.partner.clone()
        clean, failed = half(side)
        assert failed == 0
        _restore(eng, T0)
        assert np.isfinite(objective())
        sites = _poison_sites(csr.indptr.cpu().numpy(), n_fixed)
        try:
            for _, pos, bad in sites:
                csr.partner[pos] = bad
            got, failed = half(side)
            assert failed == 3
            assert all(np.isfinite(got[n]).all() for n in TABLES)
            rows = [r for r, _, _ in sites]
            for n in (side + "_feat", side + "_bias"):
                keep = np.zeros(len(got[n]), bool)
                keep[rows] = True
                assert np.array_equal(_u32(got[n])[keep], _u32(T0[n])[keep]), n
                assert np.array_equal(_u32(got[n])[~keep], _u32(clean[n])[~keep]), n
            assert not np.array_equal(_u32(clean[side + "_feat"])[rows], _u32(T0[side + "_feat"])[rows])
            assert _same(got, clean, ["mu"] + [OTHER[side] + s for s in ("_feat", "_bias")])
            if side == "user":
                _restore(eng, T0)
                assert np.isnan(objective())
        finally:
            csr.partner.copy_(clean_ids)
