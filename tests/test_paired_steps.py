"""Two Adam steps per table pass (tfr_svd_pair_bring + tfr_svd_pair_pass, SvdEngine.pair_steps) leave the state one
step per pass leaves, bit for bit: two engines from the same seed, pairing forced on and off, stepped through the same
sequence of run_stream_steps calls, are compared after every call on uint32 views (the sign of a zero counts).

The sweeps reach every (VEC, L) instantiation of adam_bring_kernel, batches whose runs start on a group edge and on a
CTA edge of that kernel, the partitioned pass (small tables), the one-grid pass over all tables in one trip and in
several trips, and every bit-neutral knob with pairing on.  The CPU tests mirror row_geom and launch_stream_chunks's
partition rule to show that, read the kernels' register use from ptxas, and check the refusals of the two entry points.
Slot-map stamps are 32 bits of global_step: the last tests restore checkpoints around 2^32 and step across it."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch

from test_geometry import NVCC, ROOT, row_geom, tuned
from tf_recomm_b200 import _lib
from tf_recomm_b200._lib import ABS_ITEM, LOSS_SIGMOID_CE, REG_BIAS, VAR_ALL, VAR_MU, VAR_UB, VAR_UF
from tf_recomm_b200.engine import TABLE_NAMES, SvdEngine, idle_slot_entry

U, I, B = 301, 203, 512
# step counts of the calls, in order: 1 to 9 and 17 steps; the calls themselves split runs of pairs
CALLS = (1, 2, 3, 4, 5, 6, 7, 8, 9, 17)
N_STEPS = sum(CALLS)
# the first call a pair: the first pair runs at global_step 0 / 1 on slot maps no step has stamped
CALLS_PAIR_FIRST = (2, 3, 1, 4)
KNOBS = ["STREAM_THREADS", "STREAM_CTAS_PER_SM", "STREAM_LD", "STREAM_ST", "STREAM_UNROLL", "STREAM_DYNAMIC", "PASS_RING",
         "PDL", "TL_EVERY_CTA", "SORT_SPLIT", "SEG_CHAIN", "SEG_TILE", "SEG_MAX_UNITS"]

SLICE_ENT, BRING_THREADS = 4, 256       # adam.cu: entries per lane group, threads per CTA of adam_bring_kernel
# the dims that reach all 12 (VEC, L) of adam_bring_kernel
BRING_DIMS = [1, 2, 3, 4, 5, 8, 9, 12, 15, 16, 17, 32, 63, 64, 128, 132, 512]
BRING_BATCHES = [1, 3, 4, 5, 31, 32, 33, 1023, 1025]
# tables the pass streams in one grid (not partitioned): (U, I, dim)
BIG_SHAPES = [(60000, 8000, 64), (60000, 8000, 132), (60000, 8000, 512), (200000, 20000, 15)]
SINGLE_TABLE_MASKS = {"uf": VAR_UF, "ub_mu": VAR_UB | VAR_MU}


def _bits(a):
    a = a.detach().contiguous().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
    return np.ascontiguousarray(a).view(np.uint32 if a.dtype.itemsize == 4 else np.uint64)


def _same_bits(a, b):
    """Two device tensors of one dtype hold the same bits (compared on the device: the big tables stay there)."""
    iv = torch.int32 if a.element_size() == 4 else torch.int64
    return a.shape == b.shape and torch.equal(a.contiguous().view(iv), b.contiguous().view(iv))


# ---- Python mirror of the pass's launch geometry ---------------------------------------------------------------------------
def pass_layout(U_, I_, d, var_mask=VAR_ALL, threads=448, ctas_per_sm=2, unroll=2, sm_count=148):
    """adam.cu: launch_stream_chunks for the two-step pass (UNROLL 2 in the kernel) over run_step's tables ->
    (partitioned, CTAs, trips of the longest-running thread)."""
    chunks = [(n, w) for bit, n, w in ((VAR_UB, U_, 1), (_lib.VAR_IB, I_, 1), (_lib.VAR_IF, I_ * d, d),
                                      (VAR_UF, U_ * d, d)) if var_mask & bit]
    units = sum((n + 3) // 4 for n, _ in chunks)
    threads = threads if 32 <= threads <= 512 else 448
    threads &= ~31
    grid = -(-units // (threads * unroll))
    cap = sm_count * ctas_per_sm
    if ctas_per_sm > 0 and grid > cap:
        grid = cap
    total = sum(n for n, _ in chunks)
    if len(chunks) > 1 and total * 12 < 32 << 20:
        return True, None, None
    trips = max(-(-(n // 4) // (grid * threads * 2)) if w % 4 == 0 else -(-n // (grid * threads)) for n, w in chunks)
    return False, grid, trips


# ---- the two engines -------------------------------------------------------------------------------------------------------
def _columns(kind, rng, sigmoid, shape=(U, I, B), n_steps=N_STEPS):
    """Training columns and the index stream (n_steps + 1 batches) of one batch pattern."""
    U_, I_, B_ = shape
    n = 4096
    users, items = rng.integers(0, U_, n), rng.integers(0, I_, n)
    idx = rng.integers(0, n, (n_steps + 1, B_))
    if kind == "repeated":          # every id of a batch occurs several times
        users, items = rng.integers(0, 23, n), rng.integers(0, 17, n)
    elif kind == "disjoint":        # batches t and t+1 share no user and no item
        half = n // 2
        users[:half], users[half:] = rng.integers(0, U_ // 2, half), rng.integers(U_ // 2, U_, n - half)
        items[:half], items[half:] = rng.integers(0, I_ // 2, half), rng.integers(I_ // 2, I_, n - half)
        idx[0::2] = rng.integers(0, half, idx[0::2].shape)
        idx[1::2] = rng.integers(half, n, idx[1::2].shape)
    elif kind == "identical":       # batch 2j+1 repeats batch 2j, and batch 2j+2 repeats 2j+1 at other positions
        idx[1::2] = idx[0::2][:idx[1::2].shape[0]]
        idx[2::2] = rng.permuted(idx[1::2][:idx[2::2].shape[0]], axis=1)
    elif kind == "hot":             # one item in most rows: its run crosses many tiles of the segment sums
        items[rng.random(n) < 0.8] = 7
    elif kind == "edges":           # runs that start on the bring kernel's group and CTA edges, and runs across them
        # batch t is rows t*B .. t*B + B - 1.  In sorted order the first half of a batch is runs of SLICE_ENT user
        # ids: every group edge, and every CTA edge k * 1024 / L below B / 2, opens a run; the rest are runs of 6, which
        # cross group edges and the CTA edge at 1024 (L = 1).  Items: runs of 8, then runs of 3 and 5 in turn, which
        # cross group edges and open a run at 1024.  A batch's run ids are a random draw of the ids, so consecutive
        # batches share rows, and the order of the positions is shuffled.
        n = (n_steps + 1) * B_
        idx = np.arange(n)
        users, items = np.empty(n, np.int64), np.empty(n, np.int64)
        for t in range(n_steps + 1):
            for col, m, r0, rest in ((users, U_, SLICE_ENT, [6]), (items, I_, 8, [3, 5])):
                lens = np.r_[np.full(B_ // 2 // r0, r0), np.tile(rest, B_ // 3 + 1)]
                runs = np.repeat(np.arange(len(lens)), lens)[:B_]
                assert runs[-1] < m
                ids = np.sort(rng.choice(m, runs[-1] + 1, replace=False))[runs]
                col[t * B_:(t + 1) * B_] = rng.permutation(ids)
    else:
        raise ValueError(kind)
    n = len(users)
    rates = (rng.random(n) < 0.5).astype(np.float32) if sigmoid else rng.integers(1, 6, n).astype(np.float32)
    return (users.astype(np.int32), items.astype(np.int32), rates), idx.reshape(-1)


def _engine(shape, d, flags, var_mask, cols, idx, pair, graph_steps, n_steps):
    U_, I_, B_ = shape
    e = SvdEngine(U_, I_, d, 0.01, 0.05, flags=flags, var_mask=var_mask, device_init_seed=5)
    e.pair_steps = pair
    e.graph_steps = graph_steps
    e.set_train_data(*cols)
    e.set_index_stream(idx, B_)
    e.set_se_ring(n_steps + 4)
    return e


def _assert_same(a, b, what):
    for n in TABLE_NAMES:
        assert _same_bits(a.t[n], b.t[n]), (what, n)
    assert set(a.slots) == set(b.slots)
    for n in a.slots:
        assert _same_bits(a.slots[n], b.slots[n]), (what, n)
    oa, ob = a.opt_scalars(), b.opt_scalars()
    for f in ("beta1_power", "beta2_power", "lr_t"):
        assert np.array_equal(_bits(np.float32([getattr(oa, f)])), _bits(np.float32([getattr(ob, f)]))), (what, f)
    for f in ("global_step", "batch_cursor"):
        assert getattr(oa, f) == getattr(ob, f), (what, f)
    assert np.array_equal(_bits(a.se_ring), _bits(b.se_ring)), (what, "se_ring")


def _run(d, kind, flags=0, var_mask=VAR_ALL, graph_steps=8, use_graph=True, seed=0, shape=(U, I, B), knobs=None,
         calls=CALLS):
    knobs = knobs or {}
    n_steps = sum(calls)
    torch.manual_seed(0)
    cols, idx = _columns(kind, np.random.default_rng(seed), bool(flags & LOSS_SIGMOID_CE), shape, n_steps)
    with tuned(**knobs):
        on = _engine(shape, d, flags, var_mask, cols, idx, True, graph_steps, n_steps)
        off = _engine(shape, d, flags, var_mask, cols, idx, False, graph_steps, n_steps)
        if "TL_EVERY_CTA" in knobs:
            on.enable_timeline()
            off.enable_timeline()
        for k, n in enumerate(calls):
            bo = on.run_stream_steps(n, use_graph=use_graph)
            bf = off.run_stream_steps(n, use_graph=use_graph)
            torch.cuda.synchronize()
            what = "%s call %d (%d steps)" % (knobs, k, n)
            for name in ("logits", "infer"):   # the call's last step
                assert np.array_equal(_bits(bo[name]), _bits(bf[name])), (what, name)
            if n >= 2:   # and the step before it, in the other buffer set (the one primed for the next call)
                po, pf = on.stream_buffers(shape[2], on._primed), off.stream_buffers(shape[2], off._primed)
                for name in ("logits", "infer"):
                    assert np.array_equal(_bits(po[name]), _bits(pf[name])), (what, "previous step", name)
            _assert_same(on, off, what)
    assert on.global_step == n_steps and on.live_slots() == 0
    on.close()
    off.close()


# ---- CPU -------------------------------------------------------------------------------------------------------------------
def test_bring_dims_reach_every_bring_instantiation():
    pairs = {(v, l) for v in (1, 4) for l in (1, 2, 4, 8, 16, 32)}
    assert {row_geom(d) for d in BRING_DIMS} == pairs, sorted(pairs - {row_geom(d) for d in BRING_DIMS})


def test_edges_batches_put_run_heads_on_group_and_cta_edges():
    """The "edges" kind: at every lane count some run of batch t+1 opens at a CTA edge of adam_bring_kernel (entry
    k * 1024 / L), some runs open on group edges (entry 4k) and some runs cross a group edge."""
    for B_ in (31, 32, 33, 1023, 1025):
        (users, items, _), idx = _columns("edges", np.random.default_rng(0), False, (U, I, B_), 3)
        heads = set()
        for col in (users, items):
            s = np.sort(col[idx[B_:2 * B_]])
            h = np.flatnonzero(np.r_[True, s[1:] != s[:-1]])
            assert np.any(h % SLICE_ENT == 0) and np.any(h % SLICE_ENT != 0), B_   # on and off group edges
            heads |= set(h.tolist())
        for lanes in (1, 2, 4, 8, 16, 32):
            cta = BRING_THREADS // lanes * SLICE_ENT
            assert any(k * cta in heads for k in range(1, -(-B_ // cta))) == (cta < B_), (B_, lanes)


def test_pass_layout_of_the_shapes():
    """Which shapes stream their tables partitioned (one slice of the grid per table), in one grid in one trip, and in
    one grid of several trips per thread (148 SMs, default knobs unless given)."""
    for d in (1, 4, 15, 64, 128, 132, 512):
        assert pass_layout(U, I, d)[0], d
    for d in BRING_DIMS:
        assert pass_layout(U, I, d)[0]
    for mask in SINGLE_TABLE_MASKS.values():   # one streamed table: never partitioned, one trip
        assert pass_layout(U, I, 64, mask) == (False, 6 if mask == VAR_UF else 1, 1)
    for U_, I_, d in BIG_SHAPES:
        part, grid, trips = pass_layout(U_, I_, d)
        assert not part and grid == 296 and trips > 1, (U_, I_, d, trips)
        part, grid, trips = pass_layout(U_, I_, d, ctas_per_sm=0)   # no cap on the grid: one trip of vector units
        assert not part and trips == (1 if d % 4 == 0 else 7)        # (the scalar path walks floats, not units)
    assert pass_layout(60000, 8000, 64)[2] == 4 and pass_layout(200000, 20000, 15)[2] == 23
    assert pass_layout(60000, 8000, 64, threads=32)[2] == 51 and pass_layout(60000, 8000, 64, ctas_per_sm=4)[2] == 2


@pytest.mark.skipif(not os.path.exists(NVCC), reason="needs the CUDA toolkit")
def test_adam_kernels_compile_without_spills(tmp_path):
    """adam.cu for sm_100a (CUDA 12.9): the 12 adam_bring_kernel instantiations (74 to 128 registers) and the two-step
    pass adam_stream_multi_kernel<2, false, 2> (64 registers, its __launch_bounds__(512, 2) budget) use no stack and do
    not spill.  <4, false, 1>, the pass of STREAM_UNROLL >= 4, does: a 176-byte stack, 544 / 596 bytes of spill stores /
    loads.  That is pinned as a bound, so a change that spills more there fails here."""
    from test_rank_users import _ptxas_lines
    obj, log = str(tmp_path / "adam.o"), str(tmp_path / "ptxas.txt")
    with open(log, "w") as f:
        subprocess.check_call([NVCC, "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-ccbin",
                               "/usr/bin/g++", "-Xcompiler", "-fPIC", "-Xptxas", "-v", "-c",
                               os.path.join(ROOT, "tf-recomm_b200", "csrc", "adam.cu"), "-o", obj],
                              stdout=f, stderr=subprocess.STDOUT)
    info = _ptxas_lines(log)
    bring = {"void tfr::adam_bring_kernel<%d, %d>" % (v, l) for v in (1, 4) for l in (1, 2, 4, 8, 16, 32)}
    pair = "void tfr::adam_stream_multi_kernel<2, false, 2>"
    assert bring | {pair} <= set(info), sorted(bring - set(info))
    for name in bring | {pair}:
        regs, stack, st, ld = info[name]
        assert (stack, st, ld) == (0, 0, 0), (name, info[name])
    assert info[pair][0] <= 64, info[pair]
    regs, stack, st, ld = info["void tfr::adam_stream_multi_kernel<4, false, 1>"]
    assert stack <= 176 and st <= 544 and ld <= 596, (regs, stack, st, ld)


def test_pair_entry_points_refuse_bad_arguments():
    """tfr_svd_pair_bring / tfr_svd_pair_pass check everything on the host before any CUDA call: SGD, row-sharded
    tables, a missing slot map or Adam slot, one workspace for both steps and B <= 0 are TFR_ERR_INVALID; a workspace
    too small for B is TFR_ERR_WORKSPACE."""
    L = _lib.load()
    dummy, d, B_ = 256, 8, 16
    need = L.tfr_svd_step_workspace_bytes(B_, d)
    assert need > 0
    t = _lib.SvdTables()
    t.user_num, t.item_num, t.dim = 4, 4, d
    for f, _ in _lib.SvdTables._fields_[4:-5]:
        setattr(t, f, dummy)

    for fn in (L.tfr_svd_pair_bring, L.tfr_svd_pair_pass):
        def call(flags=0, B=B_, ws_t=dummy, ws_n=dummy * 2, ws_t_bytes=need, ws_n_bytes=need):
            return fn(C.byref(t), dummy, B, flags, VAR_ALL, ws_t, ws_t_bytes, ws_n, ws_n_bytes, None)

        for flags in (_lib.OPT_SGD, _lib.FORK_FLAGS):
            assert call(flags=flags) == -1, (fn.__name__, flags)   # TFR_ERR_INVALID
        for B in (0, -1):
            assert call(B=B) == -1, (fn.__name__, B)
        assert call(ws_n=dummy) == -1 and call(ws_t=None) == -1 and call(ws_n=None) == -1
        for f in ("user_slot", "item_slot", "m_uf", "v_ib", "m_mu"):
            setattr(t, f, None)
            assert call() == -1, (fn.__name__, f)
            setattr(t, f, dummy)
        t.g_user_feat = t.g_item_feat = t.g_user_bias = t.g_item_bias = dummy
        assert call() == -1, fn.__name__
        t.g_user_feat = t.g_item_feat = t.g_user_bias = t.g_item_bias = None
        assert call(ws_t_bytes=need - 1) == -3 and call(ws_n_bytes=0) == -3, fn.__name__   # TFR_ERR_WORKSPACE
        t.dim = 0
        assert call() == -1, fn.__name__
        t.dim = d


STAMP_STEPS = [2 ** 32 - 3, 2 ** 32 - 2, 2 ** 32 - 1, 2 ** 32, 2 ** 33 - 1]


def test_idle_slot_entry_matches_no_upcoming_stamp():
    """The slot-map entry restore() writes carries the stamp of the step before global_step: neither global_step (a
    single step, the bring of a pair) nor global_step + 1 (a pair's table pass) matches it, modulo 2^32."""
    assert idle_slot_entry(0) == -1
    for gs in STAMP_STEPS + [0, 1, 5, 2 ** 31, 2 ** 63 - 1]:
        e = idle_slot_entry(gs)
        assert -2 ** 63 <= e < 2 ** 63
        stamp = (e >> 32) & 0xffffffff
        assert e & 0xffffffff == 0xffffffff
        assert stamp == (gs - 1) % 2 ** 32
        for k in range(2 ** 16):   # no step of the next 65536 matches it, nor the pass of a pair that ends there
            assert stamp != (gs + k) % 2 ** 32


# ---- GPU -------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module", autouse=True)
def _restore_knobs():
    saved = {k: _lib.tune_get(k) for k in KNOBS}
    try:
        yield
    finally:
        for k, v in saved.items():
            _lib.tune_set(k, v)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["repeated", "disjoint", "identical", "hot"])
@pytest.mark.parametrize("d", [1, 4, 15, 64, 128, 132, 512])
def test_pairs_match_single_steps(d, kind):
    _run(d, kind)


@pytest.mark.gpu
@pytest.mark.parametrize("d", BRING_DIMS)
def test_pairs_match_single_steps_every_bring_geometry(d):
    _run(d, "edges", seed=d, shape=(U, I, 1025), calls=(2, 3, 4))


@pytest.mark.gpu
@pytest.mark.parametrize("d", [1, 3, 17, 132])
@pytest.mark.parametrize("b", BRING_BATCHES)
def test_pairs_match_single_steps_batch_edges(d, b):
    """Batches of one entry, of one group's SLICE_ENT +- 1, of one CTA's entries at L = 32 +- 1 (d = 17, 132) and at
    L = 1 +- 1 (d = 1); d = 3 (L = 4) has its CTA edge at 256."""
    _run(d, "edges" if b >= 31 else "repeated", seed=b, shape=(U, I, b), calls=(1, 2, 3, 4))


@pytest.mark.gpu
@pytest.mark.parametrize("shape", BIG_SHAPES, ids=lambda s: "%dx%dxd%d" % s)
def test_pairs_match_single_steps_one_grid_pass(shape):
    """Tables streamed by one persistent grid in several trips per thread (test_pass_layout_of_the_shapes)."""
    U_, I_, d = shape
    _run(d, "hot", seed=3, shape=(U_, I_, 2048), calls=(1, 2, 3, 4))


@pytest.mark.gpu
@pytest.mark.parametrize("mask", list(SINGLE_TABLE_MASKS))
@pytest.mark.parametrize("d", [15, 64])
def test_pairs_match_single_steps_single_table(d, mask):
    """One streamed table (plus mu): the pass is never partitioned."""
    _run(d, "repeated", var_mask=SINGLE_TABLE_MASKS[mask], seed=4, calls=(1, 2, 3, 4))


@pytest.mark.gpu
@pytest.mark.parametrize("d", [15, 128])
def test_pairs_match_single_steps_first_call_a_pair(d):
    _run(d, "identical", seed=5, calls=CALLS_PAIR_FIRST)


PAIR_KNOBS = ([dict(STREAM_THREADS=t) for t in (32, 100, 512)] + [dict(STREAM_CTAS_PER_SM=c) for c in (0, 1, 4)] +
              [dict(STREAM_LD=h) for h in (0, 1, 2, 3)] + [dict(STREAM_ST=h) for h in (0, 1, 2, 3)] +
              [dict(PDL=1), dict(TL_EVERY_CTA=1), dict(SORT_SPLIT=1), dict(SEG_CHAIN=0)] +
              # ignored by the two-step pass, used by the single steps: ties the pair to each single-step pass variant
              [dict(STREAM_UNROLL=4), dict(STREAM_DYNAMIC=1), dict(PASS_RING=1)])


@pytest.mark.gpu
@pytest.mark.parametrize("knobs", PAIR_KNOBS, ids=lambda s: ",".join("%s=%d" % kv for kv in s.items()))
@pytest.mark.parametrize("shape", [(U, I, 128), (60000, 8000, 64)], ids=["partitioned_d128", "one_grid_d64"])
def test_pairs_match_single_steps_with_knobs(shape, knobs):
    U_, I_, d = shape
    _run(d, "hot", seed=6, shape=(U_, I_, 2048), knobs=knobs, calls=(1, 2, 3, 4))


@pytest.mark.gpu
@pytest.mark.parametrize("tile", [8, 16, 32])
@pytest.mark.parametrize("max_units", [0, 1, 2, 4])
def test_pairs_match_single_steps_seg_tile_and_units(max_units, tile):
    _run(128, "hot", seed=7, knobs=dict(SEG_TILE=tile, SEG_MAX_UNITS=max_units), calls=(1, 2, 3, 4))


@pytest.mark.gpu
@pytest.mark.parametrize("use_graph", [True, False])
@pytest.mark.parametrize("graph_steps", [2, 8])
@pytest.mark.parametrize("d", [4, 15, 128])
def test_pairs_match_single_steps_graph_and_eager(d, graph_steps, use_graph):
    _run(d, "hot", graph_steps=graph_steps, use_graph=use_graph, seed=1)


@pytest.mark.gpu
@pytest.mark.parametrize("flags,var_mask", [
    (REG_BIAS | ABS_ITEM | LOSS_SIGMOID_CE, VAR_ALL),
    (REG_BIAS, VAR_ALL & ~4),     # user features not trained
    (ABS_ITEM, VAR_ALL & ~(1 | 8)),   # bias_global and item biases not trained
    (0, 4 | 16),                  # features only
])
@pytest.mark.parametrize("d", [1, 15, 128])
def test_pairs_match_single_steps_flags_and_var_mask(d, flags, var_mask):
    _run(d, "repeated", flags=flags, var_mask=var_mask, seed=2)


@pytest.mark.gpu
def test_auto_pairs_only_where_the_pass_streams_hbm():
    small = SvdEngine(U, I, 16, 0.01, 0.05, device_init_seed=5)
    assert small._pair_steps() is False
    small.pair_steps = True
    assert small._pair_steps() is True
    sgd = SvdEngine(U, I, 16, 0.01, 0.05, flags=8, device_init_seed=5)
    sgd.pair_steps = True
    assert sgd._pair_steps() is False
    big = SvdEngine(162541, 62423, 128, 0.01, 0.05, device_init_seed=5)
    assert big._pair_steps() is True


# ---- slot-map stamps across 2^32 steps -------------------------------------------------------------------------------------
def _checkpoint(tmp_path, d):
    """A checkpoint of an engine trained a few steps (Adam slots and beta powers away from their initial values)."""
    rng = np.random.default_rng(11)
    eng = SvdEngine(U, I, d, 0.01, 0.05, device_init_seed=9)
    for _ in range(3):
        eng.train_step(rng.integers(0, U, B).astype(np.int32), rng.integers(0, I, B).astype(np.int32),
                       rng.integers(1, 6, B).astype(np.float32))
    path = str(tmp_path / "ckpt.npz")
    eng.save(path)
    return path


def _restored(tmp_path, path, d, step):
    """An engine restored from `path` with its global_step replaced by `step`."""
    with np.load(path) as z:
        arrays = {k: z[k] for k in z.files}
    arrays["__step__"] = np.array([step], np.int64)
    p = str(tmp_path / ("ckpt_%d.npz" % step))
    with open(p, "wb") as f:
        np.savez(f, **arrays)
    eng = SvdEngine(U, I, d, 0.01, 0.05, device_init_seed=1)
    eng.restore(p)
    return eng


def _assert_no_live_stamp_after_restore(tmp_path, path):
    for gs in STAMP_STEPS:
        eng = _restored(tmp_path, path, 16, gs)
        assert eng.global_step == gs
        assert eng.live_slots() == 0, (gs, eng.live_slots())
        for m in (eng.user_slot, eng.item_slot):
            stamps = ((m.cpu().numpy() >> 32) & 0xffffffff).astype(np.int64)
            assert not np.any(stamps == gs % 2 ** 32) and not np.any(stamps == (gs + 1) % 2 ** 32), gs
        eng.close()


@pytest.mark.gpu
def test_restore_leaves_no_slot_entry_an_upcoming_step_matches(tmp_path):
    """After restore() at a global_step near or past 2^32, no slot-map entry carries the stamp of the next step
    (global_step) or of a pair's pass (global_step + 1): live_slots() is 0.  Only the engine's set-up and host work
    follow the restore; no training step is run."""
    _assert_no_live_stamp_after_restore(tmp_path, _checkpoint(tmp_path, 16))


@pytest.mark.gpu
@pytest.mark.parametrize("pair", [True, False])
def test_steps_across_2_to_the_32_match_steps_at_5(tmp_path, pair):
    """One checkpoint restored at global_step 5 and at 2^32 - 3 (congruent modulo the se_ring length of 8) and stepped
    through calls of 1, 2, 3 and 2 steps: stamps wrap at 2^32 in the second engine, and training depends on global_step
    only through the stamps and the se_ring index, so both engines hold the same bits after every call."""
    d = 16
    path = _checkpoint(tmp_path, d)
    _assert_no_live_stamp_after_restore(tmp_path, path)   # stops here, before any step, if restore left a live stamp
    rng = np.random.default_rng(12)
    cols, idx = _columns("hot", rng, False, (U, I, B), 8)
    engs = []
    for gs in (5, 2 ** 32 - 3):
        e = _restored(tmp_path, path, d, gs)
        e.pair_steps = pair
        e.set_train_data(*cols)
        e.set_index_stream(idx, B)
        e.set_se_ring(8)
        engs.append(e)
    a, b = engs
    for k, n in enumerate((1, 2, 3, 2)):
        ba, bb = a.run_stream_steps(n), b.run_stream_steps(n)
        torch.cuda.synchronize()
        what = "pair=%s call %d" % (pair, k)
        for name in ("logits", "infer"):
            assert np.array_equal(_bits(ba[name]), _bits(bb[name])), (what, name)
        for n_ in TABLE_NAMES:
            assert _same_bits(a.t[n_], b.t[n_]), (what, n_)
        for n_ in a.slots:
            assert _same_bits(a.slots[n_], b.slots[n_]), (what, n_)
        oa, ob = a.opt_scalars(), b.opt_scalars()
        for f in ("beta1_power", "beta2_power", "lr_t", "lr_t_prev"):
            assert np.array_equal(_bits(np.float32([getattr(oa, f)])), _bits(np.float32([getattr(ob, f)]))), (what, f)
        assert np.array_equal(_bits(a.se_ring), _bits(b.se_ring)), (what, "se_ring")
        assert ob.global_step - oa.global_step == 2 ** 32 - 8
        assert a.live_slots() == 0 and b.live_slots() == 0
    assert b.global_step == 2 ** 32 + 5
    a.close()
    b.close()
