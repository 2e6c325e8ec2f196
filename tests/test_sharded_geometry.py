"""The row-sharded training step (BASELINE configs[4]) at every dim, world size, tile edge and tuning knob.

Both exchanges run on one GPU with G virtual ranks, as in test_gpu_parity: the all-reduce exchange is gather_owned on
every rank, a plain sum of the exchange buffers (what the NCCL all-reduce computes) and local_step on every rank; the
all-to-all exchange is _a2a_emulated_step.  Every step is compared with the single-table C oracle on the re-assembled
shards, Adam slots included, by the rules test_geometry judges the single-table step with.  Every occurrence's logits
and infer must also equal, bit for bit, what SvdEngine.forward gives on the re-assembled tables before the step: both
exchanges promise the forward kernel's arithmetic and reduction order, so a row or record sent to the wrong place cannot
hide inside a tolerance.

In row-sharded mode the segment sums read the partner rows by batch position (g_*), at a stride of dim (all-reduce) or
dim + 4 (all-to-all records) against the owner's 3 * dim, and the occurrences of rows other ranks own sort to the end
under the "not mine" key.  The sweeps below reach every segment-sum instantiation and every row geometry in that mode,
owned runs that end at a tile edge or at the not-mine boundary, a rank that receives nothing and ranks whose slice of the
batch is empty.  The CPU tests check that reach, the refusals of SGD and of tables with fewer rows than ranks, and that
the kernels of csrc/shard.cu compile without more spills than they have today.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch

import oracle
# _restore_knobs: the module-scoped autouse fixture, so every knob a test here sets leaves the module as it came in
from test_geometry import (I_SWEEP, NVCC, ROOT, SEG_TILES, SEG_UNITS, SWEEP_DIMS, U_SWEEP, _assert_state,  # noqa: F401
                           _check_outputs, _restore_knobs, _sweep_batches, row_geom, seg_cases, seg_geom, tuned)
from test_gpu_parity import _a2a_emulated_step, make_batch, zipf_ids
from tf_recomm_b200 import _lib, init, sharding
from tf_recomm_b200.engine import TABLE_NAMES

SHARD = os.path.join(ROOT, "tf-recomm_b200", "csrc", "shard.cu")
LR, REG = 1e-3, 0.05
MODELS = {"readme_adam": 0,                                   # the lean segment-sum variant
          "fork_adam": _lib.FORK_FLAGS & ~_lib.OPT_SGD}       # ABS_ITEM | sigmoid-CE | REG_BIAS: the generic variant
WORLDS, WORLD_DIMS = [1, 2, 3, 5, 8], [1, 15, 128, 260, 512]
TILE_DIMS = [15, 64, 260]
# with SWEEP_DIMS these reach, through SEG_MAX_UNITS, the instantiations no default geometry uses
SHARD_KNOB_DIMS = [2, 3, 5, 8, 12, 15, 20, 31, 33, 64, 100]
SHARD_MAX_RANKS = 8   # csrc/shard.cu: the all-to-all's layouts hold at most this many ranks

# csrc/shard.cu under CUDA 12.9, measured: (stack frame, spill stores, spill loads) in bytes of the kernels that keep
# values in local memory; every other kernel of the file keeps none.  A change that spills more fails here.
SHARD_SPILLS = {"void tfr::shard_fwd_records_kernel<4, 32>": (8, 4, 8),
                "void tfr::shard_fwd_records_kernel<4, 2>": (8, 4, 8),
                "void tfr::shard_gather_records_kernel<4, 32>": (16, 12, 12),
                "void tfr::shard_gather_records_kernel<4, 16>": (16, 12, 12),
                "void tfr::shard_gather_records_kernel<4, 8>": (16, 12, 12),
                "void tfr::shard_gather_records_kernel<4, 4>": (16, 12, 12),
                "void tfr::shard_gather_records_kernel<4, 2>": (8, 4, 4),
                "tfr::shard_bucket_finish_kernel": (8, 4, 4)}


# ---- CPU -------------------------------------------------------------------------------------------------------------------
def test_row_sharded_step_refuses_sgd():
    """With g_* set the step trains with Adam only: the SGD slice update would take the "not mine" run (key user_num /
    item_num) for a row, one past the local tables.  The refusal comes before any CUDA call; the pointers are never read.
    With a zero-byte workspace a step that is not refused stops at the workspace check, also before any CUDA call."""
    L = _lib.load()
    dummy = 256
    t = _lib.SvdTables()
    t.user_num, t.item_num, t.dim = 4, 4, 8
    for f, _ in _lib.SvdTables._fields_[4:-5]:
        setattr(t, f, dummy)
    t.g_user_feat = t.g_item_feat = t.g_user_bias = t.g_item_bias = dummy

    def step(flags):
        return L.tfr_svd_train_step(C.byref(t), dummy, dummy, dummy, dummy, 16, dummy, dummy, flags, _lib.VAR_ALL, dummy,
                                    0, None, None, 0, None)

    def presorted(flags):
        return L.tfr_svd_train_step_presorted(C.byref(t), dummy, dummy, dummy, dummy, 16, dummy, dummy, flags,
                                              _lib.VAR_ALL, 3, dummy, 0, None)

    def gathered(flags):
        return L.tfr_svd_train_step_gathered(C.byref(t), dummy, dummy, dummy, 16, flags, _lib.VAR_ALL, dummy, dummy,
                                             dummy, 0, None)

    for fn in (step, presorted, gathered):
        for flags in (_lib.OPT_SGD, _lib.FORK_FLAGS):
            assert fn(flags) == -1, (fn.__name__, flags)   # TFR_ERR_INVALID
            assert b"sgd" in L.tfr_last_error().lower(), L.tfr_last_error()
        assert fn(0) == -3, fn.__name__                     # Adam: on to the workspace check (TFR_ERR_WORKSPACE)
    t.g_user_feat = t.g_item_feat = t.g_user_bias = t.g_item_bias = None
    for fn in (step, presorted):                            # single-table SGD: on to the workspace check
        assert fn(_lib.FORK_FLAGS) == -3, fn.__name__


def test_sharded_engine_refuses_sgd():
    from tf_recomm_b200.sharded import ShardedSvdEngine
    for flags in (_lib.OPT_SGD, _lib.FORK_FLAGS):
        with pytest.raises(ValueError, match="Adam only"):
            ShardedSvdEngine(100, 50, 8, LR, REG, rank=0, world=2, flags=flags)


@pytest.mark.parametrize("U,I,G", [(257, 5, 8), (3, 131, 4), (1, 1, 2)])
def test_sharded_engine_refuses_fewer_rows_than_ranks(U, I, G):
    """A rank would own no row of a table (an empty local table); refused before anything is allocated."""
    from tf_recomm_b200.sharded import ShardedSvdEngine
    for r in (0, G - 1):
        with pytest.raises(ValueError, match="one row of each table per rank"):
            ShardedSvdEngine(U, I, 8, LR, REG, rank=r, world=G)


def test_sharded_sweeps_reach_every_geometry():
    """The dim sweep reaches every (VEC, L) the row_geom dispatchers of shard.cu (gather rows, gather records, forward
    records) and svd_forward take; with the knob sweep it reaches every segment-sum instantiation in gathered mode.
    The batches of the dim sweep at G = 3 include ranks with no user records and ranks with an empty slice."""
    pairs = {(v, l) for v in (1, 4) for l in (1, 2, 4, 8, 16, 32)}
    assert {row_geom(d) for d in SWEEP_DIMS} == pairs
    reached = {seg_geom(d) for d in SWEEP_DIMS} | {seg_geom(d, u) for d in SHARD_KNOB_DIMS for u in SEG_UNITS}
    assert reached == seg_cases(), sorted(seg_cases() - reached)
    big, one, hot = _sweep_batches(np.random.default_rng(0), U_SWEEP, I_SWEEP, False)
    assert len(set(sharding.owner(hot[0], 3))) == 1                              # two ranks get no user record
    assert [sharding.batch_slice(len(one[0]), 3, r) for r in range(3)] == [(0, 1), (1, 1), (1, 1)]   # two empty slices


@pytest.mark.skipif(not os.path.exists(NVCC), reason="needs the CUDA toolkit")
def test_shard_kernels_compile_for_every_geometry(tmp_path):
    """Every kernel of csrc/shard.cu compiles for sm_100a, at each of the twelve row geometries, within the spills
    measured above (none for the kernels not listed)."""
    from test_rank_users import _ptxas_lines
    obj, log = str(tmp_path / "shard.o"), str(tmp_path / "ptxas.txt")
    with open(log, "w") as f:
        subprocess.check_call([NVCC, "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-ccbin",
                               "/usr/bin/g++", "-Xcompiler", "-fPIC", "-Xptxas", "-v", "-c", SHARD, "-o", obj],
                              stdout=f, stderr=subprocess.STDOUT)
    info = _ptxas_lines(log)
    want = {"void tfr::%s<%d, %d>" % (k, v, l) for k in ("shard_gather_rows_kernel", "shard_gather_records_kernel",
                                                         "shard_fwd_records_kernel")
            for v in (1, 4) for l in (1, 2, 4, 8, 16, 32)}
    want |= {"tfr::" + k for k in ("shard_owner_keys_kernel", "shard_bucket_finish_kernel", "shard_fold_partials_kernel",
                                   "shard_unfold_sums_kernel", "shard_owner_prepare_kernel")}
    assert want == set(info), sorted(want ^ set(info))
    for name, (regs, stack, st, ld) in info.items():
        bound = SHARD_SPILLS.get(name, (0, 0, 0))
        assert stack <= bound[0] and st <= bound[1] and ld <= bound[2], (name, info[name])


# ---- the two exchanges on G virtual ranks, and the comparison ------------------------------------------------------------
def _allreduce_step(engs, users, items, rates):
    """gather_owned on every rank -> the sum of the exchange buffers (the all-reduce; exact, one non-zero term per
    element) -> local_step on every rank.  Every rank computes the same predictions, bit for bit."""
    e0 = engs[0].local
    B = len(users)
    du, di, dr = e0._dev_i32(users), e0._dev_i32(items), e0._dev_f32(rates)
    bufs = [e._buffers(B) for e in engs]
    for e, b in zip(engs, bufs):
        e.gather_owned(du, di, b)
    total = torch.stack([b["flat"] for b in bufs]).sum(0)
    outs = []
    for e, b in zip(engs, bufs):
        b["flat"].copy_(total)
        outs.append([x.cpu().numpy() for x in e.local_step(b, dr)])
    for r, (lg, inf) in enumerate(outs[1:], 1):
        assert np.array_equal(lg.view(np.int32), outs[0][0].view(np.int32)), "rank %d logits" % r
        assert np.array_equal(inf.view(np.int32), outs[0][1].view(np.int32)), "rank %d infer" % r
    return outs[0]


EXCHANGES = {"allreduce": _allreduce_step, "a2a": _a2a_emulated_step}


def _entry_point(name):
    """A public step of a world-1 engine (no process group), as an exchange."""
    def step(engs, users, items, rates):
        (e,) = engs
        return tuple(x.cpu().numpy() for x in getattr(e, name)(users, items, rates))
    return step


def _tables(engs):
    """The re-assembled shards as one get_tables() dict, Adam slots included.  mu and its slots: every rank holds the
    same bits (each applies the same update from the same all-reduced sum)."""
    parts = [e.local.get_tables() for e in engs]
    out = {}
    for k in parts[0]:
        if k.endswith("mu"):
            for r, p in enumerate(parts[1:], 1):
                assert np.array_equal(p[k].view(np.int32), parts[0][k].view(np.int32)), "rank %d %s" % (r, k)
            out[k] = parts[0][k]
        else:
            out[k] = sharding.unshard_table([p[k] for p in parts])
    return out


def _forward(tabs, U, I, d, flags, users, items):
    """SvdEngine.forward on one table holding the re-assembled shards."""
    from tf_recomm_b200.engine import SvdEngine
    eng = SvdEngine(U, I, d, LR, REG, flags=flags, tables=tabs)
    logits, infer = eng.forward(users, items)
    return logits.cpu().numpy(), infer.cpu().numpy()


def _sharded(G, U, I, d, flags, seed=2):
    from tf_recomm_b200.sharded import ShardedSvdEngine
    tabs = init.init_tables(U, I, d, seed=seed, bias_init="truncated_normal")
    orc = oracle.SvdOracle(tabs["mu"], tabs["user_bias"], tabs["item_bias"], tabs["user_feat"], tabs["item_feat"], LR,
                           REG, flags=flags)
    return [ShardedSvdEngine(U, I, d, LR, REG, rank=r, world=G, tables=tabs, flags=flags) for r in range(G)], orc


class _SlotMatched:
    """The oracle's state, each variable but mu moved by what the Adam steps so far take differently from the kernel's
    slots than from the oracle's: lr_t * m / (sqrt(v) + eps), summed over the steps.  Where a row's summed gradient g
    cancels to near zero (|g| down to ~1e-6 from terms of ~1e-1), that step is lr * g / (|g| + eps'), and the fp32
    rounding of g, which depends on the order of the adds, moves the variable by up to ~1e-5: more than the element
    bound, though the slots themselves still agree with the oracle's.  Judged against this state, the variable must
    follow the update its own slots give; the slots stay judged against the oracle's.  Elsewhere the shift is below
    1e-8, far inside the bound."""

    def __init__(self, orc):
        self.orc, self.shift, self.step = orc, {}, 0

    def advance(self, got):
        self.step += 1
        t = self.step
        lr_t = LR * np.sqrt(1.0 - 0.999 ** t) / (1.0 - 0.9 ** t)
        for n in TABLE_NAMES:
            if n == "mu":
                continue
            upd = [lr_t * np.asarray(sl["m_" + n], np.float64) / (np.sqrt(np.asarray(sl["v_" + n], np.float64)) + 1e-8)
                   for sl in (got, self.orc.slots)]
            self.shift[n] = self.shift.get(n, 0.0) + upd[0] - upd[1]

    def __getattr__(self, n):
        ref = getattr(self.orc, n)
        return ref if n not in self.shift else np.asarray(ref, np.float64) - self.shift[n]


def _run_sharded(G, U, I, d, flags, step, batches, what):
    """Each batch one step of `step` on G ranks: predictions bit for bit those of the forward kernel on the pre-step
    tables and within the oracle's bar, then the re-assembled slots against the oracle's and the tables against the
    oracle's moved as _SlotMatched says."""
    engs, orc = _sharded(G, U, I, d, flags)
    ref = _SlotMatched(orc)
    e_mass = 0.0
    for s, (users, items, rates) in enumerate(batches):
        at = "%s step %d (B=%d)" % (what, s, len(users))
        fwd_logits, fwd_infer = _forward(_tables(engs), U, I, d, flags, users, items)
        logits, infer = step(engs, users, items, rates)
        assert np.array_equal(logits.view(np.int32), fwd_logits.view(np.int32)), at + " logits vs forward"
        assert np.array_equal(infer.view(np.int32), fwd_infer.view(np.int32)), at + " infer vs forward"
        ref_logits, ref_infer = orc.train_step(users, items, rates)
        _check_outputs(torch.from_numpy(logits), torch.from_numpy(infer), ref_logits, ref_infer, flags, at)
        x = ref_logits.astype(np.float64)
        e = (1.0 / (1.0 + np.exp(-x)) if flags & _lib.LOSS_SIGMOID_CE else x) - rates
        e_mass += float(np.abs(e).sum())
        got = _tables(engs)
        ref.advance(got)
        _assert_state(got, ref, LR, False, at, e_mass)
        for r, e in enumerate(engs):
            assert e.local.global_step == s + 1 and e.local.live_slots() == 0, "%s rank %d" % (at, r)
    return engs


# ---- GPU: every dim, both exchanges, both kernel variants -----------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("exchange", list(EXCHANGES))
@pytest.mark.parametrize("d", SWEEP_DIMS)
@pytest.mark.parametrize("model", list(MODELS))
def test_sharded_step_every_dim_vs_oracle(model, d, exchange):
    flags = MODELS[model]
    batches = _sweep_batches(np.random.default_rng(d), U_SWEEP, I_SWEEP, bool(flags & _lib.LOSS_SIGMOID_CE))
    _run_sharded(3, U_SWEEP, I_SWEEP, d, flags, EXCHANGES[exchange], batches, "d=%d %s %s" % (d, model, exchange))


# ---- GPU: world sizes -------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("exchange", list(EXCHANGES))
@pytest.mark.parametrize("d", WORLD_DIMS)
@pytest.mark.parametrize("G", WORLDS)
def test_sharded_step_every_world_size_vs_oracle(G, d, exchange):
    batches = _sweep_batches(np.random.default_rng(100 * G + d), U_SWEEP, I_SWEEP, False)
    _run_sharded(G, U_SWEEP, I_SWEEP, d, 0, EXCHANGES[exchange], batches, "G=%d d=%d %s" % (G, d, exchange))


@pytest.mark.gpu
def test_a2a_refuses_more_ranks_than_its_layout_holds():
    from tf_recomm_b200.sharded import ShardedSvdEngine
    G = SHARD_MAX_RANKS + 1
    users, items, _ = make_batch(np.random.default_rng(9), U_SWEEP, I_SWEEP, 100)
    eng = ShardedSvdEngine(U_SWEEP, I_SWEEP, 16, LR, REG, rank=0, world=G)
    with pytest.raises(_lib.TfrError, match="invalid argument"):
        eng.a2a_bucket(users, items)
    with pytest.raises(_lib.TfrError, match="invalid argument"):
        eng.a2a_gather(eng.local._dev_i32(users[:G]), [1] * G, [0] * G)


# ---- GPU: owned runs at tile edges and at the not-mine boundary -----------------------------------------------------------
def _edge_batch(rng, n_own, n_other, hot_run=0):
    """G = 2, both sides: n_own occurrences of even ids (rank 0's rows) and n_other of odd ones, shuffled.  Sorted by
    rank 0's keys, the owned entries are [0, n_own) and the not-mine block starts at n_own; in the all-to-all receive
    buffer the owned user records come first and the item records follow, marked not-mine.  hot_run > 0: the largest
    even id takes hot_run of the owned occurrences and the others take smaller ids, so its run is the last owned one and
    ends just before the not-mine block."""
    def side(n_rows):
        evens, odds = np.arange(0, n_rows, 2), np.arange(1, n_rows, 2)
        pool = evens[:-1] if hot_run else evens
        own = np.concatenate([pool[zipf_ids(rng, len(pool), n_own - hot_run, 0.8)], np.full(hot_run, evens[-1])])
        ids = rng.permutation(np.concatenate([own, odds[zipf_ids(rng, len(odds), n_other, 0.8)]])).astype(np.int32)
        keys = np.sort(sharding.local_keys(ids, 2, 0, sharding.rows_on_rank(n_rows, 2, 0)))
        assert np.count_nonzero(ids % 2 == 0) == n_own
        if hot_run:
            assert np.all(keys[n_own - hot_run:n_own] == evens[-1] // 2) and keys[n_own - hot_run - 1] < evens[-1] // 2
        return ids
    users, items = side(U_SWEEP), side(I_SWEEP)
    return users, items, rng.integers(1, 6, len(users)).astype(np.float32)


@pytest.mark.gpu
@pytest.mark.parametrize("exchange", list(EXCHANGES))
@pytest.mark.parametrize("d", TILE_DIMS)
@pytest.mark.parametrize("tile", SEG_TILES)
def test_owned_runs_ending_at_tile_edges_vs_oracle(tile, d, exchange):
    """Rank 0 owns m*T - 1, m*T and m*T + 1 occurrences (T = SEG_TILE); then a hot owned run of 2T + 1 entries that
    crosses tiles and is the last owned run, its end at, just before and just after a tile edge."""
    rng = np.random.default_rng(1000 * tile + d)
    batches = [_edge_batch(rng, m * tile + dl, tile + 5) for m in (1, 4) for dl in (-1, 0, 1)]
    batches += [_edge_batch(rng, 3 * tile + dl, tile + 5, hot_run=2 * tile + 1) for dl in (-1, 0, 1)]
    with tuned(SEG_TILE=tile):
        _run_sharded(2, U_SWEEP, I_SWEEP, d, 0, EXCHANGES[exchange], batches, "T=%d d=%d %s" % (tile, d, exchange))


# ---- GPU: idle ranks and empty slices ----------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("exchange", list(EXCHANGES))
@pytest.mark.parametrize("d", [15, 128])
def test_rank_that_receives_nothing_takes_the_adam_step(d, exchange):
    """G = 2 and batches of even ids only: rank 1 owns no occurrence (all-to-all: it receives no record, the n = 0 path
    of tfr_svd_train_step_gathered), yet every one of its rows takes the Adam step the oracle takes (m and v decay, the
    row moves by the decayed m).  A mixed batch first gives rank 1's rows non-zero slots."""
    rng = np.random.default_rng(d)
    evens = [(u - u % 2, i - i % 2, r) for u, i, r in (make_batch(rng, U_SWEEP, I_SWEEP, B) for B in (500, 1, 300))]
    batches = [make_batch(rng, U_SWEEP, I_SWEEP, 500)] + evens + [make_batch(rng, U_SWEEP, I_SWEEP, 200)]
    engs = _run_sharded(2, U_SWEEP, I_SWEEP, d, 0, EXCHANGES[exchange], batches, "even ids d=%d %s" % (d, exchange))
    assert engs[1].local.global_step == len(batches)


@pytest.mark.gpu
@pytest.mark.parametrize("exchange", list(EXCHANGES))
@pytest.mark.parametrize("G", [5, 8])
def test_batches_smaller_than_the_world_vs_oracle(G, exchange):
    """B < G: the ranks past the batch draw an empty slice (n = 0 in tfr_shard_bucket and tfr_shard_fwd_records)."""
    rng = np.random.default_rng(G)
    batches = [make_batch(rng, U_SWEEP, I_SWEEP, B) for B in (1, 2, G - 1, G, G + 1, 3 * G - 1)]
    assert sharding.batch_slice(1, G, G - 1) == (1, 1)
    _run_sharded(G, U_SWEEP, I_SWEEP, 15, 0, EXCHANGES[exchange], batches, "G=%d %s" % (G, exchange))


# ---- GPU: SEG_TILE x SEG_MAX_UNITS in gathered mode ----------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("exchange", list(EXCHANGES))
@pytest.mark.parametrize("d", SHARD_KNOB_DIMS)
@pytest.mark.parametrize("max_units", SEG_UNITS)
@pytest.mark.parametrize("tile", SEG_TILES)
def test_sharded_seg_tile_and_units_vs_oracle(tile, max_units, d, exchange):
    batches = _sweep_batches(np.random.default_rng(2000 + d), U_SWEEP, I_SWEEP, False)
    with tuned(SEG_TILE=tile, SEG_MAX_UNITS=max_units):
        _run_sharded(3, U_SWEEP, I_SWEEP, d, 0, EXCHANGES[exchange], batches,
                     "d=%d tile=%d units=%d %s" % (d, tile, max_units, exchange))


# ---- GPU: the public entry points at world = 1 -----------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("entry", ["train_step", "train_step_from_slices", "train_step_a2a"])
@pytest.mark.parametrize("d", [15, 128])
@pytest.mark.parametrize("model", list(MODELS))
def test_public_entry_points_at_world_one_vs_oracle(model, d, entry):
    flags = MODELS[model]
    rng = np.random.default_rng(d)
    binary = bool(flags & _lib.LOSS_SIGMOID_CE)
    batches = _sweep_batches(rng, U_SWEEP, I_SWEEP, binary) + [make_batch(rng, U_SWEEP, I_SWEEP, 700, binary)]
    _run_sharded(1, U_SWEEP, I_SWEEP, d, flags, _entry_point(entry), batches, "%s d=%d %s" % (entry, d, model))


@pytest.mark.gpu
@pytest.mark.parametrize("d", [15, 128])
def test_a2a_next_slice_and_emulation_keep_every_bit(d):
    """train_step_a2a with next_slice (the next step's plan made on the side stream under this step's pass) gives the
    same bits as the same steps without it, and at G = 1 both equal the emulated exchange of the GPU tests."""
    rng = np.random.default_rng(d)
    batches = [make_batch(rng, U_SWEEP, I_SWEEP, B) for B in (1500, 1, 400, 999)]
    runs = {}
    for mode in ("next_slice", "plain", "emulated"):
        (eng,), _ = _sharded(1, U_SWEEP, I_SWEEP, d, 0)
        dev = [(eng.local._dev_i32(u), eng.local._dev_i32(i), r) for u, i, r in batches]
        outs = []
        for s, (u, i, r) in enumerate(dev):
            if mode == "emulated":
                out = _a2a_emulated_step([eng], *batches[s])
            else:
                nxt = dev[s + 1][:2] if mode == "next_slice" and s + 1 < len(dev) else None
                out = tuple(x.cpu().numpy() for x in eng.train_step_a2a(u, i, r, next_slice=nxt))
                if nxt is not None:
                    assert eng._plan["key"][0] is dev[s + 1][0]    # the next step takes this plan, not a new one
            outs.append((out, _tables([eng])))
        runs[mode] = outs
    for mode in ("next_slice", "emulated"):
        for s, (((lg, inf), tabs), ((lg0, inf0), tabs0)) in enumerate(zip(runs[mode], runs["plain"])):
            assert np.array_equal(lg.view(np.int32), lg0.view(np.int32)), "%s step %d logits" % (mode, s)
            assert np.array_equal(inf.view(np.int32), inf0.view(np.int32)), "%s step %d infer" % (mode, s)
            assert set(tabs) == set(tabs0)
            for k in tabs:
                assert np.array_equal(tabs[k].view(np.int32), tabs0[k].view(np.int32)), "%s step %d %s" % (mode, s, k)
