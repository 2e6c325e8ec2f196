"""The chain tiles kernel (csrc/chain.cu) at every geometry it is instantiated for, bit for bit against the kernel it
replaces.

chain_tiles_kernel<L, T> runs the fused forward + segment sums of the README model (plain dot, Adam) where the default
geometry is (VEC 4, L lanes, 4 units) and (L, T) is one of TFR_CHAIN_CASES; it claims to compute exactly what
segsum_tiles_kernel<4, L, 4, true, false> computes.  SEG_CHAIN=0 sends the same launches to that kernel, so every GPU
test below runs one engine with each and compares on uint32 views (the sign of a zero counts): the logits and infer of
the first step, its per-CTA and folded partial sums, the summed gradients at the run heads of both sides and both slot
maps, then every table, Adam slot and step scalar after three steps.  The CPU tests read the case list out of chain.cu,
check with test_geometry's mirror of seg_geom / seg_tile that the sweep reaches every case and every case's grid-stride
loop (one lane group walking more than one tile), and that the kernels compile without spills.
"""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

from test_geometry import NVCC, ROOT, _run_vs_oracle, seg_cases, seg_geom, seg_tile, tuned, zipf_ids
from tf_recomm_b200 import _lib
from tf_recomm_b200._lib import LOSS_SIGMOID_CE, REG_BIAS, VAR_ALL, VAR_UB, VAR_UF
from tf_recomm_b200.engine import TABLE_NAMES

CHAIN = os.path.join(ROOT, "tf-recomm_b200", "csrc", "chain.cu")
SEG_THREADS = 128
# the dim sweep, per lane count: (dim, SEG_MAX_UNITS).  100 = 25 units, 4 per lane over 8 lanes: lane 0 holds four
# units, lane 1 four, ..., the last units absent on most lanes; 132 = 33 units over 16 lanes: lane 0 alone has a third
CHAIN_DIMS = {8: [(128, 0), (100, 4)], 16: [(132, 0), (192, 0), (256, 0)], 32: [(260, 0), (384, 0), (512, 0)]}
CHAIN_TILES = [8, 16, 32]
U_CH, I_CH = 2003, 1009
LR, REG = 1e-3, 0.05


def chain_cases():
    """The (L, T) list of TFR_CHAIN_CASES in csrc/chain.cu."""
    line = next(s for s in open(CHAIN).read().split("\n") if s.startswith("#define TFR_CHAIN_CASES(X)"))
    cases = [tuple(int(x) for x in m) for m in re.findall(r"X\((\d+), (\d+)\)", line)]
    assert len(cases) == len(set(cases))
    return set(cases)


def chain_case(d, max_units, tile, flags=0):
    """segsum.cu: launch_segsum's choice for the fused step at a forced tile -- the (L, T) of chain_tiles_kernel, or
    None where segsum_tiles_kernel runs."""
    vec, lanes, units = seg_geom(d, max_units)
    if flags & (_lib.ABS_ITEM | _lib.OPT_SGD) or (vec, units) != (4, 4) or (lanes, tile) not in chain_cases():
        return None
    return lanes, tile


def stride_threshold(lanes):
    """Tiles a grid of MAX_PARTIALS CTAs of SEG_THREADS / L lane groups covers in one trip: past it, groups stride."""
    return _lib.MAX_PARTIALS * (SEG_THREADS // lanes)


def batch_sizes(lanes, tile):
    """Batch sizes of the sweep at one geometry (the kinds of _batch)."""
    return {"b1": 1, "t_minus_1": tile - 1, "t": tile, "t_plus_1": tile + 1, "two_t_plus_1": 2 * tile + 1,
            "zipf": 64 * tile, "mid": 12 * tile, "one_user": 10 * tile + 3,
            "stride": stride_threshold(lanes) * tile + 1}


BATCH_KINDS = list(batch_sizes(8, 8))


def _sweep():
    """(dim, max_units, tile) of the GPU sweep that take the chain kernel."""
    return [(d, u, t) for L in CHAIN_DIMS for d, u in CHAIN_DIMS[L] for t in CHAIN_TILES if chain_case(d, u, t)]


# ---- CPU -------------------------------------------------------------------------------------------------------------------
def test_chain_cases_are_segment_sum_cases():
    cases = chain_cases()
    assert len(cases) == 8
    assert {(4, L, 4) for L, _ in cases} <= seg_cases()
    assert {T for _, T in cases} <= set(CHAIN_TILES)


def test_sweep_reaches_every_chain_case_and_its_grid_stride_loop():
    cases = chain_cases()
    reached = {chain_case(d, u, t) for d, u, t in _sweep()}
    assert reached == cases, sorted(cases ^ reached)
    for d, u, t in _sweep():
        L, T = chain_case(d, u, t)
        n_tiles = -(-batch_sizes(L, T)["stride"] // T)
        assert n_tiles == stride_threshold(L) + 1
    # every lane count of the sweep is the geometry the dims are listed under
    for L, dims in CHAIN_DIMS.items():
        for d, u in dims:
            assert seg_geom(d, u) == (4, L, 4), (d, u)
    # <8, 32> is dropped: the old kernel serves it, and every non-chain geometry
    assert chain_case(128, 0, 32) is None and chain_case(100, 4, 32) is None
    assert chain_case(128, 0, 16, _lib.ABS_ITEM) is None and chain_case(128, 0, 16, _lib.OPT_SGD) is None
    assert chain_case(100, 0, 16) is None   # 25 units at the default geometry: 32 lanes of one unit
    assert chain_case(15, 0, 16) is None and chain_case(128, 1, 16) is None
    # <16, 32> is the default geometry of dims 132..256 once the batch is large (148 SMs)
    for d in (132, 192, 256):
        assert chain_case(d, 0, seg_tile(65536, d, 0, 148)) == (16, 32), d
    assert chain_case(128, 0, seg_tile(65536, 128, 0, 148)) == (8, 16)


@pytest.mark.skipif(not os.path.exists(NVCC), reason="needs the CUDA toolkit")
def test_chain_kernels_compile_without_spills(tmp_path):
    """The eight chain_tiles_kernel instantiations compile for sm_100a with no stack and no spills (CUDA 12.9: 110 to
    112 registers under __launch_bounds__(128, 4))."""
    from test_rank_users import _ptxas_lines
    obj, log = str(tmp_path / "chain.o"), str(tmp_path / "ptxas.txt")
    with open(log, "w") as f:
        subprocess.check_call([NVCC, "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-ccbin",
                               "/usr/bin/g++", "-Xcompiler", "-fPIC", "-Xptxas", "-v", "-c", CHAIN, "-o", obj],
                              stdout=f, stderr=subprocess.STDOUT)
    info = _ptxas_lines(log)
    want = {"void tfr::chain_tiles_kernel<%d, %d>" % c for c in chain_cases()}
    assert want == set(info), sorted(want ^ set(info))
    for name, (regs, stack, st, ld) in info.items():
        assert (stack, st, ld) == (0, 0, 0), (name, info[name])
        assert regs <= 128, (name, regs)   # four CTAs of 128 threads per SM


# ---- GPU -------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module", autouse=True)
def _restore_knobs():
    saved = {k: _lib.tune_get(k) for k in ("SEG_CHAIN", "SEG_TILE", "SEG_MAX_UNITS")}
    try:
        yield
    finally:
        for k, v in saved.items():
            _lib.tune_set(k, v)


def _crosses(ids, tile):
    """Some run of equal ids in sorted order crosses a tile boundary."""
    s = np.sort(ids)
    edges = np.arange(tile, len(s), tile)
    return bool(np.any(s[edges] == s[edges - 1]))


def _batch(kind, rng, lanes, tile, binary=False):
    B = batch_sizes(lanes, tile)[kind]
    users, items = zipf_ids(rng, U_CH, B, 0.6), zipf_ids(rng, I_CH, B, 1.0)
    if kind == "zipf":        # hot ids on both sides: runs that cross tiles on both sides
        users, items = zipf_ids(rng, U_CH, B, 1.1), zipf_ids(rng, I_CH, B, 1.2)
        assert _crosses(users, tile) and _crosses(items, tile)
    elif kind == "mid":       # a run of 5T + 3 entries on each side: at least three whole tiles (TILE_MID)
        users[:5 * tile + 3] = users[0]
        items[-(5 * tile + 3):] = items[-1]
    elif kind == "one_user":  # one run over the whole batch on the user side
        users[:] = users[0]
    rates = rng.integers(0, 2, B).astype(np.float32) if binary else rng.integers(1, 6, B).astype(np.float32)
    return users, items, rates


_TABLES = {}


def _engine(d, reg, flags, var_mask):
    from tf_recomm_b200 import init
    from tf_recomm_b200.engine import SvdEngine
    if d not in _TABLES:
        _TABLES[d] = init.init_tables(U_CH, I_CH, d, seed=d, bias_init="truncated_normal")
    return SvdEngine(U_CH, I_CH, d, LR, reg, flags=flags, var_mask=var_mask, tables=_TABLES[d])


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint32 if a.dtype.itemsize == 4 else np.uint64)


def _first_step(eng, batch):
    """One training step; what its fused segment sums left: logits, infer, the per-CTA and folded partial sums, the
    summed gradients at the run heads of both sides, both slot maps."""
    import torch
    users, items, rates = batch
    B, d = len(users), eng.d
    logits, infer = eng.train_step(users, items, rates)
    torch.cuda.synchronize()
    ws, wbase = eng.step_ws(B), eng.workspace(B)

    def ws_arr(ptr, count, dtype):
        off = ptr - wbase.data_ptr()
        return wbase[off:off + count * np.dtype(dtype).itemsize].cpu().numpy().view(dtype).copy()

    n = _lib.load().tfr_svd_fused_n_partials(d, B)
    assert 1 <= n <= _lib.MAX_PARTIALS
    res = {"logits": logits.cpu().numpy(), "infer": infer.cpu().numpy(),
           "user_slot": eng.user_slot.cpu().numpy(), "item_slot": eng.item_slot.cpu().numpy()}
    for name, ptr, dt in (("partials", ws.partials, np.float32), ("se_partials", ws.se_partials, np.float64)):
        p = ws_arr(ptr, _lib.MAX_PARTIALS + 1, dt)
        res[name] = p[:n]
        res[name + "_folded"] = p[_lib.MAX_PARTIALS:]
    for side, sid_p, gs_p, gsb_p in (("user", ws.su_ids, ws.gsum_uf, ws.gsum_ub),
                                     ("item", ws.si_ids, ws.gsum_if, ws.gsum_ib)):
        sid = ws_arr(sid_p, B, np.int32)
        heads = np.flatnonzero(np.r_[True, sid[1:] != sid[:-1]])
        res[side + "_sums"] = ws_arr(gs_p, B * d, np.float32).reshape(B, d)[heads]
        res[side + "_bias_sums"] = ws_arr(gsb_p, B, np.float32)[heads]
    return res


def _run(d, max_units, tile, batches, reg=REG, flags=0, var_mask=VAR_ALL):
    """Steps a fresh engine through `batches` with the chain kernel and with the old one; returns both sides'
    first-step outputs and final states."""
    out = {}
    for chain in (1, 0):
        with tuned(SEG_CHAIN=chain, SEG_TILE=tile, SEG_MAX_UNITS=max_units):
            eng = _engine(d, reg, flags, var_mask)
            first = _first_step(eng, batches[0])
            for b in batches[1:]:
                eng.train_step(*b)
            out[chain] = first, eng.get_tables(), eng.opt_scalars(), eng.live_slots()
    return out


def _assert_same(out, what):
    (f1, t1, s1, l1), (f0, t0, s0, l0) = out[1], out[0]
    assert set(f1) == set(f0)
    for k in f1:
        assert f1[k].shape == f0[k].shape and np.array_equal(_bits(f1[k]), _bits(f0[k])), (what, "first step", k)
    assert set(t1) == set(t0) and set(TABLE_NAMES) <= set(t1)
    for k in t1:
        assert np.array_equal(_bits(t1[k]), _bits(t0[k])), (what, k)
    for f in ("global_step", "beta1_power", "beta2_power", "lr_t", "lr_t_prev", "g_mu", "se_sum"):
        assert np.array_equal(_bits(np.array([getattr(s1, f)])), _bits(np.array([getattr(s0, f)]))), (what, f)
    assert l1 == l0 == 0


def _batches(kind, seed, lanes, tile, binary=False, steps=3):
    rng = np.random.default_rng(seed)
    return [_batch(kind, rng, lanes, tile, binary) for _ in range(steps)]


@pytest.mark.gpu
@pytest.mark.parametrize("d,max_units,tile", _sweep(), ids=lambda v: str(v))
def test_chain_kernel_matches_segsum_tiles_kernel(d, max_units, tile):
    """Every batch kind at every (dim, tile) of the sweep: the edges of a tile (B = 1, T - 1, T, T + 1, 2T + 1), runs
    across tiles on both sides, runs over three or more whole tiles, one user in every entry, and a batch one tile past
    the grid-stride threshold (every lane group of a full grid walks a second tile, the first group a third)."""
    L, T = chain_case(d, max_units, tile)
    for k, kind in enumerate(BATCH_KINDS):
        batches = _batches(kind, 100 * d + 10 * tile + k, L, T)
        _assert_same(_run(d, max_units, tile, batches), "d=%d tile=%d %s" % (d, tile, kind))


# one dim per lane count, each at every chain tile: the eight cases
CASE_DIMS = [(128, 0, 8), (128, 0, 16), (132, 0, 8), (256, 0, 16), (192, 0, 32), (260, 0, 8), (512, 0, 16), (384, 0, 32)]
FLAG_SETS = {"reg_bias": (REG_BIAS, VAR_ALL), "sigmoid_ce": (LOSS_SIGMOID_CE, VAR_ALL),
             "reg_bias_sigmoid_ce": (REG_BIAS | LOSS_SIGMOID_CE, VAR_ALL),
             "partial_var_mask": (0, VAR_ALL & ~(VAR_UF | VAR_UB))}


def test_case_dims_cover_every_chain_case():
    assert {chain_case(d, u, t) for d, u, t in CASE_DIMS} == chain_cases()


@pytest.mark.gpu
@pytest.mark.parametrize("flag_set", list(FLAG_SETS))
@pytest.mark.parametrize("d,max_units,tile", CASE_DIMS, ids=lambda v: str(v))
def test_chain_kernel_matches_with_every_flag_that_takes_it(d, max_units, tile, flag_set):
    flags, var_mask = FLAG_SETS[flag_set]
    assert chain_case(d, max_units, tile, flags)
    L, T = chain_case(d, max_units, tile)
    for k, kind in enumerate(("zipf", "two_t_plus_1", "mid")):
        batches = _batches(kind, 7 * d + tile + k, L, T, binary=bool(flags & LOSS_SIGMOID_CE))
        _assert_same(_run(d, max_units, tile, batches, flags=flags, var_mask=var_mask),
                     "d=%d tile=%d %s %s" % (d, tile, flag_set, kind))


@pytest.mark.gpu
@pytest.mark.parametrize("d,max_units,tile", CASE_DIMS, ids=lambda v: str(v))
def test_chain_kernel_matches_on_signed_zeros(d, max_units, tile):
    """reg = 0 and every rating the exact fp32 logit of its entry: e = 0 for every entry, so every gradient term is a
    signed zero (-0 where both the partner's and the own row's element are negative).  The logits are those of a step
    on the same fresh tables."""
    L, T = chain_case(d, max_units, tile)
    users, items, _ = _batch("zipf", np.random.default_rng(d + tile), L, T)
    with tuned(SEG_CHAIN=0, SEG_TILE=tile, SEG_MAX_UNITS=max_units):
        logits, _ = _engine(d, 0.0, 0, VAR_ALL).train_step(users, items, np.zeros(len(users), np.float32))
    batch = (users, items, logits.cpu().numpy())
    out = _run(d, max_units, tile, [batch], reg=0.0)
    _assert_same(out, "d=%d tile=%d signed zeros" % (d, tile))
    first = out[1][0]
    assert np.array_equal(_bits(first["logits"]), _bits(batch[2]))
    for side in ("user", "item"):
        s = first[side + "_sums"]
        assert not np.any(s), side   # all zeros
    assert np.all(first["partials"] == 0) and np.all(first["se_partials"] == 0)


@pytest.mark.gpu
@pytest.mark.parametrize("d,tile", [(132, 16), (132, 32), (256, 16), (256, 32)])
def test_chain_l16_cases_keep_oracle_parity(d, tile):
    """<16, 16> and <16, 32> against the C oracle (test_geometry's SEG_TILE sweep does not reach 16 lanes at four
    units): 132 gives lane 0 a third unit, 256 fills all four units of every lane."""
    assert chain_case(d, 0, tile) == (16, tile)
    with tuned(SEG_TILE=tile, SEG_MAX_UNITS=0):
        _run_vs_oracle(d, 0, 2000 + d + tile, "d=%d tile=%d" % (d, tile))
