"""Two Adam steps per table pass (tfr_svd_pair_bring + tfr_svd_pair_pass, SvdEngine.pair_steps) leave the state one
step per pass leaves, bit for bit: two engines from the same seed, pairing forced on and off, stepped through the same
sequence of run_stream_steps calls, are compared after every call on uint32 views (the sign of a zero counts)."""
import numpy as np
import pytest
import torch

from tf_recomm_b200._lib import ABS_ITEM, LOSS_SIGMOID_CE, REG_BIAS, VAR_ALL
from tf_recomm_b200.engine import TABLE_NAMES, SvdEngine

U, I, B = 301, 203, 512
# step counts of the calls, in order: 1 to 9 and 17 steps; the calls themselves split runs of pairs
CALLS = (1, 2, 3, 4, 5, 6, 7, 8, 9, 17)
N_STEPS = sum(CALLS)


def _bits(a):
    a = a.detach().contiguous().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
    return np.ascontiguousarray(a).view(np.uint32 if a.dtype.itemsize == 4 else np.uint64)


def _columns(kind, rng, sigmoid):
    """Training columns and the index stream (N_STEPS + 1 batches) of one batch pattern."""
    n = 4096
    users, items = rng.integers(0, U, n), rng.integers(0, I, n)
    idx = rng.integers(0, n, (N_STEPS + 1, B))
    if kind == "repeated":          # every id of a batch occurs several times
        users, items = rng.integers(0, 23, n), rng.integers(0, 17, n)
    elif kind == "disjoint":        # batches t and t+1 share no user and no item
        half = n // 2
        users[:half], users[half:] = rng.integers(0, U // 2, half), rng.integers(U // 2, U, n - half)
        items[:half], items[half:] = rng.integers(0, I // 2, half), rng.integers(I // 2, I, n - half)
        idx[0::2] = rng.integers(0, half, idx[0::2].shape)
        idx[1::2] = rng.integers(half, n, idx[1::2].shape)
    elif kind == "identical":       # batch 2j+1 repeats batch 2j, and batch 2j+2 repeats 2j+1 at other positions
        idx[1::2] = idx[0::2][:idx[1::2].shape[0]]
        idx[2::2] = rng.permuted(idx[1::2][:idx[2::2].shape[0]], axis=1)
    elif kind == "hot":             # one item in most rows: its run crosses many tiles of the segment sums
        items[rng.random(n) < 0.8] = 7
    else:
        raise ValueError(kind)
    rates = (rng.random(n) < 0.5).astype(np.float32) if sigmoid else rng.integers(1, 6, n).astype(np.float32)
    return (users.astype(np.int32), items.astype(np.int32), rates), idx.reshape(-1)


def _engine(d, flags, var_mask, cols, idx, pair, graph_steps):
    e = SvdEngine(U, I, d, 0.01, 0.05, flags=flags, var_mask=var_mask, device_init_seed=5)
    e.pair_steps = pair
    e.graph_steps = graph_steps
    e.set_train_data(*cols)
    e.set_index_stream(idx, B)
    e.set_se_ring(N_STEPS + 4)
    return e


def _assert_same(a, b, what):
    for n in TABLE_NAMES:
        assert np.array_equal(_bits(a.t[n]), _bits(b.t[n])), (what, n)
    for n in a.slots:
        assert np.array_equal(_bits(a.slots[n]), _bits(b.slots[n])), (what, n)
    oa, ob = a.opt_scalars(), b.opt_scalars()
    for f in ("beta1_power", "beta2_power", "lr_t"):
        assert np.array_equal(_bits(np.float32([getattr(oa, f)])), _bits(np.float32([getattr(ob, f)]))), (what, f)
    for f in ("global_step", "batch_cursor"):
        assert getattr(oa, f) == getattr(ob, f), (what, f)
    assert np.array_equal(_bits(a.se_ring), _bits(b.se_ring)), (what, "se_ring")


def _run(d, kind, flags=0, var_mask=VAR_ALL, graph_steps=8, use_graph=True, seed=0):
    torch.manual_seed(0)
    cols, idx = _columns(kind, np.random.default_rng(seed), bool(flags & LOSS_SIGMOID_CE))
    on = _engine(d, flags, var_mask, cols, idx, True, graph_steps)
    off = _engine(d, flags, var_mask, cols, idx, False, graph_steps)
    for k, n in enumerate(CALLS):
        bo = on.run_stream_steps(n, use_graph=use_graph)
        bf = off.run_stream_steps(n, use_graph=use_graph)
        torch.cuda.synchronize()
        what = "call %d (%d steps)" % (k, n)
        for name in ("logits", "infer"):   # the call's last step
            assert np.array_equal(_bits(bo[name]), _bits(bf[name])), (what, name)
        if n >= 2:   # and the step before it, in the other buffer set (the one primed for the next call)
            po, pf = on.stream_buffers(B, on._primed), off.stream_buffers(B, off._primed)
            for name in ("logits", "infer"):
                assert np.array_equal(_bits(po[name]), _bits(pf[name])), (what, "previous step", name)
        _assert_same(on, off, what)
    assert on.global_step == N_STEPS
    on.close()
    off.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["repeated", "disjoint", "identical", "hot"])
@pytest.mark.parametrize("d", [1, 4, 15, 64, 128, 132, 512])
def test_pairs_match_single_steps(d, kind):
    _run(d, kind)


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
