"""Alternating least squares at the ML-25M shape (162541 x 62423, dim 128, reg = config.LAMBDA_REG): SvdEngine.als_data /
als_sweep / training_objective on the synthetic training split (synthetic.make_ratings at the ml25m shape, ~22.5 M ratings),
tables drawn on the device with device_init_seed as tools/fold_in_bench.py does (Adam layout, as the driver trains).

Reports, in one JSON line (the GPU's name and power limit are read in the same run):
  - plan: als_data from host arrays to a ready plan (both CSRs, both row lists), host clock around a device synchronise;
  - per sweep (CUDA events over warmed-up calls): the user half-sweep, the item half-sweep, the objective / mu step, and the
    whole sweep; the kernels' own times (torch.profiler, a run of its own): chunked Gram, combine + solve of heavy rows,
    light rows, per side, and the objective;
  - the FP64 rate of each half-sweep from the FLOP count 2 (sum_rows n (D (D + 1) / 2 + D) + rows (D^3 / 6 + D^2)),
    D = dim + 1 (the count tools/fold_in_bench.py uses), against the data sheet's 37 TFLOP/s for one B200 of an HGX B200 (a
    data-sheet figure, not a measurement);
  - an ALS_CHUNK sweep (1024 .. 16384): plan chunks, workspace, half-sweep times;
  - the training objective, training RMSE and validation RMSE after each of 10 sweeps from the device initialisation.
Usage (GPU box): python tools/als_bench.py [--out FILE] [--sweeps N]"""
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import tf_recomm_b200  # noqa: E402,F401
from tf_recomm_b200 import _lib, config, synthetic  # noqa: E402
from tf_recomm_b200.engine import SvdEngine  # noqa: E402
from recommend_bench import FP64_DATASHEET, gpu_info, timed  # noqa: E402

CHUNKS = (1024, 2048, 4096, 8192, 16384)
# the half-sweep kernels are one template for ALS and iALS: their profiler names carry the form of the system
FORMS = (("FiForm<true, false, true> >", "FiRatings>"), ("FiForm<false, true, false> >", "FiImplicit>"))


def kernel_label(key):
    """A profiler event's kernel name without its parameters: 'als_objective_rows_kernel',
    'half_sweep_rows_kernel<FiRatings>', 'half_sweep_rows_kernel<FiImplicit>', ..."""
    name = key.split("(")[0].replace("void ", "").replace("tfr::", "")
    for form, label in FORMS:
        name = name.replace(form, label)
    return name


def flops(counts, dim):
    D = dim + 1
    nz = counts[counts > 0]
    return 2.0 * (float(np.sum(nz, dtype=np.float64)) * (D * (D + 1) / 2 + D) + len(nz) * (D ** 3 / 6 + D ** 2))


def halves(eng, data, reg):
    T = eng.t
    user = lambda: eng._half_sweep(data, reg, data.by_user, data.user_plan, (T["item_feat"], T["item_bias"], eng.I),  # noqa: E731
                                   (T["user_feat"], T["user_bias"]))
    item = lambda: eng._half_sweep(data, reg, data.by_item, data.item_plan, (T["user_feat"], T["user_bias"], eng.U),  # noqa: E731
                                   (T["item_feat"], T["item_bias"]))
    mu = lambda: eng._objective(data, reg, T["mu"].data_ptr())  # noqa: E731
    return user, item, mu


def plan_info(data):
    return dict(chunk=data.chunk, workspace_mb=data.workspace.numel() / 2 ** 20,
                **{side + "_" + k: int(getattr(p, k).numel()) for side, p in (("user", data.user_plan),
                                                                               ("item", data.item_plan))
                   for k in ("light", "heavy", "chunk_heavy")})


def kernel_times(eng, data, reg, reps=3):
    """Per-kernel device time (ms per sweep) from torch.profiler over `reps` sweeps, the two half-sweeps apart."""
    from torch.profiler import ProfilerActivity, profile
    user, item, mu = halves(eng, data, reg)
    out = {}
    for label, fn in (("user", user), ("item", item), ("objective", mu)):
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(reps):
                fn()
            torch.cuda.synchronize()
        for ev in prof.key_averages():
            if "als_" in ev.key or "half_sweep_" in ev.key:
                name = kernel_label(ev.key)
                dt = getattr(ev, "device_time_total", None)
                if dt is None:
                    dt = ev.cuda_time_total
                out["%s.%s" % (label, name)] = dt / 1e3 / reps
    return out


def main():
    out_path = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else None
    n_sweeps = int(sys.argv[sys.argv.index("--sweeps") + 1]) if "--sweeps" in sys.argv else 10
    name, power = gpu_info()
    reg = config.LAMBDA_REG
    res = dict(gpu=name, power_limit=power, reg=reg, fp64_datasheet_tflops=FP64_DATASHEET / 1e12)
    U, I, N = synthetic.SHAPES["ml25m"]
    d = 128
    users, items, rates = synthetic.make_ratings(U, I, N, seed=config.SEED)
    (tu, ti, tr), (vu, vi, vr) = synthetic.split(users, items, rates)
    del users, items, rates
    eng = SvdEngine(U, I, d, config.LEARNING_RATE, reg, device_init_seed=3)
    cu, ci = np.bincount(tu, minlength=U), np.bincount(ti, minlength=I)
    res["shape"] = dict(users=U, items=I, dim=d, train_ratings=int(len(tu)), val_ratings=int(len(vu)),
                        user_count_max=int(cu.max()), item_count_max=int(ci.max()),
                        items_over_4096=int((ci > 4096).sum()), their_ratings=int(ci[ci > 4096].sum()))
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    data = eng.als_data(tu, ti, tr)
    torch.cuda.synchronize()
    res["plan_build_ms"] = (time.perf_counter() - t0) * 1e3
    res["plan"] = plan_info(data)
    fl_u, fl_i = flops(cu, d), flops(ci, d)
    # ---- 10 sweeps from the initialisation: objective, train and validation RMSE after each --------------------------------
    vu_d, vi_d = torch.from_numpy(vu.astype(np.int32)).cuda(), torch.from_numpy(vi.astype(np.int32)).cuda()
    vr_d = torch.from_numpy(vr.astype(np.float32)).cuda()

    def val_rmse():
        _, inf = eng.forward(vu_d, vi_d)
        return float(torch.sqrt(torch.mean((inf.double() - vr_d.double()) ** 2)))
    obj = eng.training_objective(data)
    curve = [dict(sweep=0, loss=obj["loss"], train_rmse=obj["rmse"], val_rmse=val_rmse())]
    for s in range(1, n_sweeps + 1):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        failed = eng.als_sweep(data)
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) * 1e3
        obj = eng.training_objective(data)
        curve.append(dict(sweep=s, sweep_ms=dt, loss=obj["loss"], train_rmse=obj["rmse"], val_rmse=val_rmse(),
                          failed=int(failed.item())))
        print(json.dumps(curve[-1]), file=sys.stderr)
    res["curve"] = curve
    # ---- per-sweep phases (CUDA events, warmed up) ---------------------------------------------------------------------------
    user, item, mu = halves(eng, data, reg)
    ms_u, _ = timed(user, 5)
    ms_i, _ = timed(item, 5)
    ms_mu, _ = timed(mu, 20)
    ms_sweep, _ = timed(lambda: eng.als_sweep(data), 3)
    res["phases_ms"] = dict(user_half=ms_u, item_half=ms_i, objective_mu=ms_mu, sweep=ms_sweep)
    res["fp64"] = dict(user_flop=fl_u, item_flop=fl_i, user_tflops=fl_u / (ms_u * 1e-3) / 1e12,
                       item_tflops=fl_i / (ms_i * 1e-3) / 1e12,
                       user_fraction_of_datasheet=fl_u / (ms_u * 1e-3) / FP64_DATASHEET,
                       item_fraction_of_datasheet=fl_i / (ms_i * 1e-3) / FP64_DATASHEET,
                       sweep_fraction_of_datasheet=(fl_u + fl_i) / (ms_sweep * 1e-3) / FP64_DATASHEET)
    res["kernels_ms_per_call"] = kernel_times(eng, data, reg)
    # ---- ALS_CHUNK sweep ------------------------------------------------------------------------------------------------------
    default = _lib.tune_get("ALS_CHUNK")
    rows = []
    for c in CHUNKS:
        _lib.tune_set("ALS_CHUNK", c)
        del data
        torch.cuda.empty_cache()
        data = eng.als_data(tu, ti, tr)
        user, item, _ = halves(eng, data, reg)
        r = dict(plan_info(data), user_half_ms=timed(user, 3)[0], item_half_ms=timed(item, 3)[0])
        rows.append(r)
        print(json.dumps(r), file=sys.stderr)
    _lib.tune_set("ALS_CHUNK", default)
    res["als_chunk_default"] = default
    res["als_chunk_sweep"] = rows
    line = json.dumps(res)
    print(line)
    if out_path:
        os.makedirs(os.path.dirname(out_path) or ".", exist_ok=True)
        with open(out_path, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
