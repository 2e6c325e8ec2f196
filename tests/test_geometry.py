"""The training step at every kernel geometry and tuning knob.

The segment sums (csrc/segsum.cu) run one of the (VEC, L, UNITS) instantiations of segsum_tiles_kernel that seg_geom picks
from the dim and SEG_MAX_UNITS; the forward, the SGD slice update and the shard gathers pick a (VEC, L) from row_geom
(csrc/common.cuh).  The CPU tests mirror both functions, read the instantiation list out of segsum.cu and check that
every dim of 1..512 has an instantiation and that the GPU sweeps below reach every one of them.  The GPU tests compare
the step with the C oracle at each geometry, and the tuning knobs with a default-knob run: bit for bit where a knob only
changes launch geometry, at the oracle's 1e-5 bar where it moves fp32 rounding (include/tfrecomm.h lists which is which).
"""
import ctypes as C
import os
import re
import subprocess
from contextlib import contextmanager

import numpy as np
import pytest

from test_gpu_parity import RTOL, assert_fp32_close, both, gpu_sort, make_batch, zipf_ids
from tf_recomm_b200 import _lib
from tf_recomm_b200.engine import TABLE_NAMES

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NVCC = "/usr/local/cuda/bin/nvcc"
SEGSUM = os.path.join(ROOT, "tf-recomm_b200", "csrc", "segsum.cu")

# the dim sweep against the oracle: with the default geometry these reach every (VEC, L, UNITS) that any dim reaches,
# and every row_geom (VEC, L)
SWEEP_DIMS = [1, 2, 3, 4, 5, 7, 8, 12, 15, 16, 17, 24, 31, 32, 36, 48, 63, 64, 65, 96, 100, 127, 128, 129, 132, 160, 191,
              192, 255, 256, 257, 260, 384, 511, 512]
# the SEG_TILE x SEG_MAX_UNITS sweep: with forced unit counts these reach the instantiations no default geometry uses
KNOB_DIMS = [2, 3, 5, 8, 12, 15, 20, 31, 33, 64, 100, 128, 191, 260]
SEG_TILES = [8, 16, 32]
SEG_UNITS = [0, 1, 2, 4]
SWEEP_FLAGS = {"readme_adam": 0,                               # the lean fused variant
               "fork_sgd": _lib.FORK_FLAGS,                    # the generic variant and the SGD slice update
               "abs_regbias_adam": _lib.ABS_ITEM | _lib.REG_BIAS}  # the generic fused variant
KNOBS = ["SEG_TILE", "SEG_MAX_UNITS", "SMEM_CARVEOUT", "TILES_CARVEOUT", "STREAM_LD", "STREAM_ST", "STREAM_CTAS_PER_SM",
         "STREAM_UNROLL", "STREAM_THREADS", "STREAM_DYNAMIC", "TL_EVERY_CTA", "PDL", "SORT_SPLIT", "PASS_RING",
         "RING_SLOT_MODE", "RING_L2_HINT"]


# ---- Python mirror of the host-side geometry ------------------------------------------------------------------------------
def seg_cases():
    """The (VEC, L, UNITS) list of TFR_SEG_CASES in csrc/segsum.cu."""
    lines = open(SEGSUM).read().split("\n")
    start = next(k for k, s in enumerate(lines) if s.startswith("#define TFR_SEG_CASES(X)"))
    body = []
    for s in lines[start:]:
        body.append(s)
        if not s.rstrip().endswith("\\"):
            break
    cases = [tuple(int(x) for x in m) for m in re.findall(r"X\((\d+), (\d+), (\d+)\)", "\n".join(body))]
    assert len(cases) == len(set(cases))
    return set(cases)


def _seg_geom_max_units(dim, forced):
    vec = 4 if dim % 4 == 0 else 1
    n = dim // vec
    max_units = forced or (4 if n >= 32 else 1)
    lanes = 1
    while lanes * max_units < n and lanes < 32:
        lanes <<= 1
    u = -(-n // lanes)
    return vec, lanes, next((r for r in (1, 2, 4, 8, 16) if u <= r), u)


def seg_geom(dim, max_units=0):
    """segsum.cu: seg_geom with SEG_MAX_UNITS = max_units."""
    forced = max_units if max_units in (1, 2, 4) else 0
    g = _seg_geom_max_units(dim, forced)
    if forced and g not in seg_cases():
        g = _seg_geom_max_units(dim, 0)
    return g


def seg_tile(B, dim, max_units, sm_count):
    """segsum.cu: seg_tile with SEG_TILE = 0."""
    groups_per_warp = 32 // seg_geom(dim, max_units)[1]
    for tile in (32, 16):
        if (2 * -(-B // tile) + groups_per_warp - 1) // groups_per_warp >= sm_count * 12:
            return tile
    return 8


def segsum_grid_x(dim, B, max_units, tile):
    """segsum.cu: segsum_grid_x = tfr_svd_fused_n_partials."""
    n_tiles = (B + tile - 1) // tile
    groups_per_cta = 128 // seg_geom(dim, max_units)[1]
    return max(1, min((n_tiles + groups_per_cta - 1) // groups_per_cta, _lib.MAX_PARTIALS))


def row_geom(dim):
    """common.cuh: row_geom."""
    vec = 4 if dim % 4 == 0 else 1
    lanes = 1
    while lanes < dim // vec and lanes < 32:
        lanes <<= 1
    return vec, lanes


@contextmanager
def tuned(**settings):
    """Sets knobs for the body of the with-statement, then puts back what they were."""
    saved = {k: _lib.tune_get(k) for k in settings}
    try:
        for k, v in settings.items():
            _lib.tune_set(k, v)
        yield
    finally:
        for k, v in saved.items():
            _lib.tune_set(k, v)


@pytest.fixture(scope="module", autouse=True)
def _restore_knobs():
    """Whatever a test of this module does, every knob it can touch leaves the module as it came in."""
    saved = {k: _lib.tune_get(k) for k in KNOBS}
    try:
        yield
    finally:
        for k, v in saved.items():
            _lib.tune_set(k, v)


# ---- CPU -------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("max_units", SEG_UNITS)
def test_every_dim_up_to_512_has_a_segment_sum_instantiation(max_units):
    cases = seg_cases()
    assert len(cases) == 31
    missing = [d for d in range(1, 513) if seg_geom(d, max_units) not in cases]
    assert not missing, missing
    assert seg_geom(513, max_units) not in cases and seg_geom(516, max_units) not in cases   # the documented limit


@pytest.mark.parametrize("max_units", SEG_UNITS)
def test_geometry_mirror_matches_the_library(max_units):
    """The mirror above is the library's: tfr_svd_fused_n_partials (the fused forward's partial count, which needs no
    device) is a function of the lanes seg_geom picks and the tile seg_tile picks, for every dim of 1..512.  A forced unit
    count without an instantiation must fall back to the default geometry in seg_geom itself, or the partial count (and the
    tile size of the workspace) would disagree with the launch."""
    L = _lib.load()
    n = L.tfr_device_sm_count()
    sm = n if n > 0 else 148   # the library's own assumption without a device
    with tuned(SEG_MAX_UNITS=max_units, SEG_TILE=32):
        B = 32 * 128 * 32      # 4096 tiles of 32: 32 * lanes partials
        for d in range(1, 513):
            assert L.tfr_svd_fused_n_partials(d, B) == segsum_grid_x(d, B, max_units, 32), d
    with tuned(SEG_MAX_UNITS=max_units, SEG_TILE=0):
        for B in (1500, 300000, 2000000):
            for d in range(1, 513, 7):
                t = seg_tile(B, d, max_units, sm)
                assert L.tfr_svd_fused_n_partials(d, B) == segsum_grid_x(d, B, max_units, t), (d, B)


def test_sweeps_reach_every_instantiation_and_row_geometry():
    cases = seg_cases()
    by_default = {seg_geom(d) for d in SWEEP_DIMS}
    assert by_default == {seg_geom(d) for d in range(1, 513)}, sorted({seg_geom(d) for d in range(1, 513)} - by_default)
    forced = {seg_geom(d, u) for d in KNOB_DIMS for u in SEG_UNITS}
    assert by_default | forced == cases, sorted(cases - by_default - forced)
    pairs = {(v, l) for v in (1, 4) for l in (1, 2, 4, 8, 16, 32)}
    assert {row_geom(d) for d in SWEEP_DIMS} == pairs, sorted(pairs - {row_geom(d) for d in SWEEP_DIMS})


@pytest.mark.skipif(not os.path.exists(NVCC), reason="needs the CUDA toolkit")
def test_segment_sum_kernels_compile_for_every_case(tmp_path):
    """All 124 segsum_tiles_kernel variants (31 cases x fused / unfused x lean / generic) and both fix-up kernels compile
    for sm_100a.  CUDA 12.9: the tiles kernels use 54 to 168 registers ((1, 32, 16): 123 to 168; (1, 32, 8): 96 to 128),
    both fix-up kernels 80 (__launch_bounds__(256, 3)).  They are not spill-free: 28 of the 126 kernels keep values in
    local memory.  18 of them, fixup<4> included, park one 8-byte value that is written at entry and read at exit (the
    debug-timeline pointer of TlScope); the other 10 park 16 to 48 bytes, the most in the fused lean (1, 8, 2) and (1, 32, 2)
    and the fused generic (4, 32, 1) variants.  The bound below is that measured worst case: a new case or a change that
    spills more fails here."""
    from test_rank_users import _ptxas_lines
    obj, log = str(tmp_path / "segsum.o"), str(tmp_path / "ptxas.txt")
    with open(log, "w") as f:
        subprocess.check_call([NVCC, "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-ccbin",
                               "/usr/bin/g++", "-Xcompiler", "-fPIC", "-Xptxas", "-v", "-c", SEGSUM, "-o", obj],
                              stdout=f, stderr=subprocess.STDOUT)
    info = _ptxas_lines(log)
    want = {"void tfr::segsum_tiles_kernel<%d, %d, %d, %s, %s>" % (v, l, u, fu, ge)
            for v, l, u in seg_cases() for fu in ("false", "true") for ge in ("false", "true")}
    want |= {"void tfr::segsum_fixup_kernel<1>", "void tfr::segsum_fixup_kernel<4>"}
    assert want == set(info), sorted(want ^ set(info))
    for name, (regs, stack, st, ld) in info.items():
        assert stack <= 24 and st <= 48 and ld <= 72, (name, info[name])


# ---- GPU: the dim sweep against the C oracle ---------------------------------------------------------------------------------
U_SWEEP, I_SWEEP = 257, 131


def _sweep_batches(rng, U, I, binary):
    """A Zipf batch whose runs cross tiles on both sides, a batch of one entry, and a batch whose every entry is one user
    (a run of hundreds of tiles: the fix-up's long-chain path)."""
    hot = make_batch(rng, U, I, 400, binary)
    hot = (np.full(400, rng.integers(U), np.int32), hot[1], hot[2])
    return [make_batch(rng, U, I, 1500, binary), make_batch(rng, U, I, 1, binary), hot]


def _check_outputs(logits, infer, ref_logits, ref_infer, flags, what):
    logits, infer = logits.cpu().numpy(), infer.cpu().numpy()
    np.testing.assert_allclose(logits, ref_logits, rtol=RTOL, atol=2e-6, err_msg=what)
    if flags & _lib.LOSS_SIGMOID_CE:
        diff = infer != ref_infer   # round(sigmoid(x)) may flip only where sigmoid is within float error of 0.5
        assert np.all(np.abs(ref_logits[diff]) < 1e-5), what
    else:
        np.testing.assert_allclose(infer, ref_infer, rtol=RTOL, atol=1e-6, err_msg=what)


def _assert_state(got, orc, lr, sgd, what, e_mass):
    """test_gpu_parity.assert_state_close, with the slot allowance it gives long runs (a hot row's slots are a ~400-term
    sum in tile order against the oracle's one-after-the-other order), except for the scalar mu.  Its update is one sum
    over the batch, sum_b e_b, which cancels in the fork's loss (e = sigmoid(x) - z, about +-0.5 each): mu is judged
    against the mass of its terms, lr * sum_b |e_b| accumulated over the steps (e_mass).  got: the tables and Adam slots
    as SvdEngine.get_tables() gives them (one engine's, or re-assembled shards); sgd: the model has no slots."""
    for n in TABLE_NAMES:
        ref = getattr(orc, n)
        if n == "mu":
            err = abs(float(got[n][0]) - float(ref[0]))
            assert err <= RTOL * abs(float(ref[0])) + RTOL * lr * e_mass, "%s mu: |error| %.3g" % (what, err)
        else:
            assert_fp32_close(got[n], ref, "%s %s" % (what, n), max_abs=4 * lr + 1e-6)
        if not sgd:
            for s in ("m_", "v_"):
                assert_fp32_close(got[s + n], orc.slots[s + n], "%s %s%s" % (what, s, n), rtol=5e-5)


def _run_vs_oracle(d, flags, seed, what):
    rng = np.random.default_rng(seed)
    sgd = bool(flags & _lib.OPT_SGD)
    eng, orc = both(U_SWEEP, I_SWEEP, d, 5e-3 if sgd else 1e-3, 0.01 if sgd else 0.05, flags=flags)
    e_mass = 0.0
    for s, (users, items, rates) in enumerate(_sweep_batches(rng, U_SWEEP, I_SWEEP, bool(flags & _lib.LOSS_SIGMOID_CE))):
        logits, infer = eng.train_step(users, items, rates)
        ref_logits, ref_infer = orc.train_step(users, items, rates)
        _check_outputs(logits, infer, ref_logits, ref_infer, flags, "%s step %d" % (what, s))
        x = ref_logits.astype(np.float64)
        e = (1.0 / (1.0 + np.exp(-x)) if flags & _lib.LOSS_SIGMOID_CE else x) - rates
        e_mass += float(np.abs(e).sum())
        _assert_state(eng.get_tables(), orc, eng.hyper["lr"], eng.sgd, "%s step %d" % (what, s), e_mass)
    assert eng.global_step == 3 and eng.live_slots() == 0


@pytest.mark.gpu
@pytest.mark.parametrize("d", SWEEP_DIMS)
@pytest.mark.parametrize("model", list(SWEEP_FLAGS))
def test_train_step_every_dim_vs_oracle(d, model):
    _run_vs_oracle(d, SWEEP_FLAGS[model], d, "d=%d %s" % (d, model))


# ---- GPU: knobs that move fp32 rounding keep oracle parity ------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("d", KNOB_DIMS)
@pytest.mark.parametrize("max_units", SEG_UNITS)
@pytest.mark.parametrize("tile", SEG_TILES)
def test_seg_tile_and_units_keep_oracle_parity(d, max_units, tile):
    with tuned(SEG_TILE=tile, SEG_MAX_UNITS=max_units):
        _run_vs_oracle(d, 0, 1000 + d, "d=%d tile=%d units=%d" % (d, tile, max_units))


def _unfused_segment_sums(d, users, items, rates):
    """tfr_svd_fwd_err -> id sort -> tfr_svd_segment_grads (the generic, unfused tiles kernel + fix-up) on a fresh engine:
    the summed gradients at the run heads, both sides."""
    import torch
    L = _lib.load()
    U, I, B = U_SWEEP, I_SWEEP, len(users)
    eng, _ = both(U, I, d, 1e-3, 0.05)
    du, di, dr = eng._dev_i32(users), eng._dev_i32(items), eng._dev_f32(rates)
    ws = eng.step_ws(B)
    st = torch.cuda.current_stream().cuda_stream
    out = torch.empty(2, B, device="cuda")
    tp = C.byref(eng.tables_struct)
    _lib.check(L.tfr_svd_begin_step(eng.opt.data_ptr(), st))
    _lib.check(L.tfr_svd_fwd_err(tp, eng.opt.data_ptr(), du.data_ptr(), di.data_ptr(), dr.data_ptr(), B,
                                 out[0].data_ptr(), out[1].data_ptr(), C.byref(ws), st))
    _lib.check(L.tfr_dedup_sort_pairs(du.data_ptr(), U, ws.su_ids, ws.su_pos, di.data_ptr(), I, ws.si_ids, ws.si_pos,
                                      B, ws.sort_ws, ws.sort_ws_bytes, st))
    _lib.check(L.tfr_svd_segment_grads(tp, eng.opt.data_ptr(), du.data_ptr(), di.data_ptr(), B, C.byref(ws), st))
    torch.cuda.synchronize()
    wbase = eng.workspace(B)

    def ws_arr(ptr, count, dtype):
        off = ptr - wbase.data_ptr()
        return wbase[off:off + count * np.dtype(dtype).itemsize].cpu().numpy().view(dtype)

    res = {}
    for side, sid_p, gs_p, gsb_p in (("user", ws.su_ids, ws.gsum_uf, ws.gsum_ub), ("item", ws.si_ids, ws.gsum_if, ws.gsum_ib)):
        sid = ws_arr(sid_p, B, np.int32)
        heads = np.flatnonzero(np.r_[True, sid[1:] != sid[:-1]])
        res[side] = ws_arr(gs_p, B * d, np.float32).reshape(B, d)[heads].copy()
        res[side + "_bias"] = ws_arr(gsb_p, B, np.float32)[heads].copy()
    return res


@pytest.mark.gpu
@pytest.mark.parametrize("d", KNOB_DIMS)
@pytest.mark.parametrize("tile", SEG_TILES)
def test_unfused_segment_sums_do_not_depend_on_lanes(d, tile):
    """At a fixed tile, each column of a run adds its entries in batch order whatever the lanes per row are: the unfused
    sums are bit-identical across SEG_MAX_UNITS (only the fused forward's dot product depends on L)."""
    rng = np.random.default_rng(d + tile)
    users, items, rates = make_batch(rng, U_SWEEP, I_SWEEP, 1500)
    users[:300] = users[0]   # one run of 300: a long chain at every tile size
    got = {}
    for u in SEG_UNITS:
        with tuned(SEG_TILE=tile, SEG_MAX_UNITS=u):
            got[u] = _unfused_segment_sums(d, users, items, rates)
    for u in SEG_UNITS[1:]:
        for k in got[0]:
            assert np.array_equal(got[u][k].view(np.int32), got[0][k].view(np.int32)), (u, k)


# ---- GPU: knobs that change launch geometry only keep every bit ---------------------------------------------------------------
BIT_SHAPES = {"small_d15": (257, 131, 15), "small_d64": (257, 131, 64),   # the partitioned pass: floats * 12 < 32 Mi
              "large_d64": (60000, 8000, 64)}                               # one grid over all four tables
BIT_STEPS, BIT_B = 4, 2000
BIT_SETTINGS = ([dict(STREAM_THREADS=t) for t in (32, 64, 96, 100, 256, 512)] +
                [dict(STREAM_CTAS_PER_SM=c) for c in (0, 1, 4)] +
                [dict(STREAM_UNROLL=u) for u in (0, 1, 4)] +
                [dict(STREAM_DYNAMIC=1), dict(STREAM_DYNAMIC=1, STREAM_THREADS=100), dict(STREAM_DYNAMIC=1, STREAM_UNROLL=4)] +
                [dict(STREAM_LD=h) for h in (0, 1, 2, 3)] + [dict(STREAM_ST=h) for h in (0, 1, 2, 3)] +
                [dict(TL_EVERY_CTA=1), dict(SORT_SPLIT=1), dict(PDL=1)] +
                [dict(SMEM_CARVEOUT=c) for c in (0, 100)] + [dict(TILES_CARVEOUT=c) for c in (0, 100)] +
                [dict(PASS_RING=1, RING_SLOT_MODE=m) for m in (0, 1, 2)] +
                [dict(PASS_RING=1, RING_L2_HINT=h) for h in (0, 1, 2, 3)])
_BIT_REF = {}


def _bit_run(shape, timeline=False):
    U, I, d = BIT_SHAPES[shape]
    rng = np.random.default_rng(U + d)
    eng, _ = both(U, I, d, 1e-3, 0.05)
    if timeline:
        eng.enable_timeline()
    outs = []
    for _ in range(BIT_STEPS):
        logits, infer = eng.train_step(*make_batch(rng, U, I, BIT_B))
        outs.append((logits.cpu().numpy(), infer.cpu().numpy()))
    return outs, eng.get_tables(), eng.opt_scalars()


def _assert_bits_equal(a, b, what):
    (oa, ta, sa), (ob, tb, sb) = a, b
    for s, ((la, ia), (lb, ib)) in enumerate(zip(oa, ob)):
        assert np.array_equal(la.view(np.int32), lb.view(np.int32)), "%s logits step %d" % (what, s)
        assert np.array_equal(ia.view(np.int32), ib.view(np.int32)), "%s infer step %d" % (what, s)
    assert set(ta) == set(tb)
    for n in ta:
        assert np.array_equal(ta[n].view(np.int32), tb[n].view(np.int32)), "%s %s" % (what, n)
    for f in ("global_step", "beta1_power", "beta2_power", "lr_t", "g_mu", "se_sum"):
        assert getattr(sa, f) == getattr(sb, f), "%s %s" % (what, f)


@pytest.mark.gpu
@pytest.mark.parametrize("settings", BIT_SETTINGS, ids=lambda s: ",".join("%s=%d" % kv for kv in s.items()))
@pytest.mark.parametrize("shape", list(BIT_SHAPES))
def test_geometry_knobs_keep_every_bit(shape, settings):
    if shape not in _BIT_REF:
        _BIT_REF[shape] = _bit_run(shape)
    with tuned(**settings):
        got = _bit_run(shape, timeline="TL_EVERY_CTA" in settings)
    _assert_bits_equal(_BIT_REF[shape], got, "%s %s" % (shape, settings))


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 2, 31, 32, 33, 511, 512, 513, 1000, 10000, 65536, 200001])
def test_split_sort_bit_exact(n):
    """SORT_SPLIT=1 (one launch per phase) sorts exactly as test_dedup_sort_bit_exact's one-launch form."""
    rng = np.random.default_rng(n)
    max_a, max_b = 162541, 3952
    ids_a, ids_b = zipf_ids(rng, max_a, n, 0.8), zipf_ids(rng, max_b, n, 1.1)
    with tuned(SORT_SPLIT=1):
        sa, pa, sb, pb = gpu_sort(ids_a, max_a, ids_b, max_b)
    for ids, s, p in ((ids_a, sa, pa), (ids_b, sb, pb)):
        order = np.argsort(ids, kind="stable").astype(np.int32)
        assert np.array_equal(p.cpu().numpy(), order)
        assert np.array_equal(s.cpu().numpy(), ids[order])


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(500, 300, 15), (3000, 1500, 128)])
def test_pdl_graph_steps_keep_every_bit(shape):
    """PDL=1 in captured graphs (run_stream_steps, pipelined and plain) and in eager stream steps: the same bits as without."""
    import torch
    U, I, d = shape
    B, N, steps = 1024, 20000, 10
    rng = np.random.default_rng(d)
    cu, ci = zipf_ids(rng, U, N, 0.6), zipf_ids(rng, I, N, 1.0)
    cr = rng.integers(1, 6, N).astype(np.float32)
    row_index = rng.integers(0, N, steps * B)
    out = {}
    for pdl in (0, 1):
        with tuned(PDL=pdl):
            for mode in ("pipelined", "plain", "eager"):
                eng, _ = both(U, I, d, 1e-3, 0.05)
                eng.set_train_data(cu, ci, cr)
                eng.set_index_stream(row_index, B)
                bufs = eng.run_stream_steps(steps, use_graph=mode != "eager", pipeline=mode == "pipelined")
                torch.cuda.synchronize()
                out[pdl, mode] = ([(bufs["logits"].cpu().numpy(), bufs["infer"].cpu().numpy())], eng.get_tables(),
                                  eng.opt_scalars())
    for mode in ("pipelined", "plain", "eager"):
        _assert_bits_equal(out[0, mode], out[1, mode], "PDL %s" % mode)
    assert out[1, "pipelined"][2].global_step == steps
