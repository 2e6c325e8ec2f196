"""bench.py -- the driver's measurement contract for the TF-recomm hot path (matrix-factorization train step).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch: batch assembly -> forward + d cost/d logits -> id dedup
(radix sort + ordered segment sums) -> TF-semantics sparse Adam over the WHOLE tables.  README model (squared
error + L2 + Adam), fp32.  Prints ONE JSON line (rank 0).

Workloads (BASELINE.json configs):
  ml25m_d128_b65536   configs[3], default at N=1: 162541 x 62423, dim 128, batch 65536 -- the configuration on which
                      the metric's "HBM GB/s frac of peak" is defined (BASELINE.md section 4) and the largest one
                      that fits one GPU; its 765 MB/step working set is larger than the 126 MB L2, so no flush is
                      needed between timed steps.
  ml1m_d15_b10000     configs[1] (README speed-tuning shape); launch/L2-bound, reported under "also" at N=1.
  ml1m_d15_b1000      configs[0] shape.
  sharded_100Mx10M    configs[4], N >= 2: tables + Adam state row-sharded (id mod N), strong scaling.

`value` = ratings/s with the training columns and the pre-drawn index stream resident in HBM, each step one replay
of a captured CUDA graph, timed with CUDA events.  `e2e` = the same metric through the host-fed call
(Session.run's path: pinned host batch -> H2D -> step -> D2H of the fetched predictions), copies inside the
timed region.  `roofline` = the dominant kernel (adam_stream_multi_kernel, the whole-table pass) timed live with
CUDA events around its launches.  `cpu_baseline` / `--impl reference` = the CPU restatement of the TF path
(oracle/tfr_oracle.c, OpenMP over all host cores) on a bounded sample -- the reference's own code cannot run here
(TensorFlow absent, ops.py does not import; DESIGN.md).

--steps K sets the timed steps of `value` and of `e2e`.  `e2e`'s timed region includes the fill of its feed pipeline (the
first three batches are handed over inside it), a share of the time that grows as K shrinks: compare e2e numbers taken
at the same K.  --dump-outputs DIR writes what the last timed step of `value`
computed as DIR/<name>.npy (float32, about 5 MB): see last_step_outputs.  Columns, initial tables and index stream are
all seeded, so two builds run with the same arguments can be compared array for array.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    "ml25m_d128_b65536": dict(U=162541, I=62423, N=25000095, d=128, B=65536, config="configs[3]"),
    "ml1m_d15_b10000": dict(U=6040, I=3952, N=1000209, d=15, B=10000, config="configs[1]"),
    "ml1m_d15_b1000": dict(U=6040, I=3952, N=1000209, d=15, B=1000, config="configs[0]"),
}
LR, REG = 1e-3, 0.05
README_EPOCH_S = {"ml1m_d15_b1000": 4.1, "ml1m_d15_b10000": 1.1}   # README.md:51-57,63 (unspecified hardware)
PUBLISHED_RATINGS_PER_S = {"ml1m_d15_b10000": 0.82e6}              # BASELINE.md section 1 (derived from README.md:63)


def algorithmic_bytes_step(U, I, d, B):
    """SURVEY 8d / BASELINE.md section 4: Adam read+write of var,m,v over both tables incl. biases + one gather of
    each side's row+bias + ids and rating."""
    return 24 * (U + I) * (d + 1) + 8 * B * (d + 1) + 12 * B


def make_columns(w, seed=13575):
    """Synthetic rating columns of the workload's shape (log-normal user activity, Zipf item popularity, ratings
    1..5); 90/10 split like the README run -> the train part."""
    rng = np.random.default_rng(seed)
    n = int(round(w["N"] * 0.9))
    act = rng.lognormal(0.0, 1.0, w["U"])
    pop = 1.0 / np.arange(1, w["I"] + 1)
    users = rng.choice(w["U"], size=n, p=act / act.sum()).astype(np.int32)
    items = rng.permutation(w["I"])[rng.choice(w["I"], size=n, p=pop / pop.sum())].astype(np.int32)
    rates = rng.integers(1, 6, n).astype(np.float32)
    return users, items, rates


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        super().__init__(daemon=True)
        self.gpu_index, self.rows, self.proc = gpu_index, [], None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([x.strip() for x in line.split(",")])
        except Exception:
            pass

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
        self.join(timeout=2)
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(len(r) >= 7 and r[3 + k].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(self.rows[0][1]), "reasons": reasons,
                "samples": len(sm)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p))["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ---------------------------------------------------------------------------------------------------------------
def cpu_reference_run(w, steps, warmup, seed=13575):
    """The CPU restatement of the TF path on the workload's shape, all host cores (OpenMP)."""
    import oracle
    from tf_recomm_b200 import init
    rng = np.random.default_rng(seed)
    tabs = init.init_tables(w["U"], w["I"], w["d"], seed=seed)
    orc = oracle.SvdOracle(tabs["mu"], tabs["user_bias"], tabs["item_bias"], tabs["user_feat"], tabs["item_feat"], LR, REG)
    act = rng.lognormal(0.0, 1.0, w["U"]); act /= act.sum()
    pop = 1.0 / np.arange(1, w["I"] + 1); pop /= pop.sum()
    perm = rng.permutation(w["I"])
    B = w["B"]
    times = []
    for s in range(warmup + steps):
        users = rng.choice(w["U"], size=B, p=act).astype(np.int32)
        items = perm[rng.choice(w["I"], size=B, p=pop)].astype(np.int32)
        rates = rng.integers(1, 6, B).astype(np.float32)
        t0 = time.perf_counter()
        orc.train_step(users, items, rates)
        if s >= warmup:
            times.append(time.perf_counter() - t0)
    return float(np.sum(times)), len(times)


def workload_config(name, w):
    """The `config` object of BOTH arms (ours and --impl reference): the same keys and values, so that the driver's
    same_config comparison holds.  Arm-specific remarks live in top-level `notes`."""
    bytes_step = algorithmic_bytes_step(w["U"], w["I"], w["d"], w["B"])
    return {"workload": name, "baseline_config": w["config"], "users": w["U"], "items": w["I"], "dim": w["d"],
            "batch": w["B"], "ratings": w["N"], "model": "README: squared error + L2 + Adam (TF IndexedSlices semantics)",
            "lr": LR, "reg": REG,
            "l2_policy": ("per-step working set %.0f MB > 126 MB L2: no flush needed" % (bytes_step / 1e6))
            if bytes_step > 126e6 else
            ("working set %.1f MB is L2-resident by construction (launch-bound config)" % (bytes_step / 1e6))}


def reference_arm(args, w, name):
    cores = os.cpu_count()
    steps = args.steps
    warm = max(args.warmup, 3)    # the same warm-up rule as our arm
    tot, n = cpu_reference_run(w, steps, warm)
    ms = tot / n * 1e3
    val = w["B"] / (tot / n)
    line = {
        "impl": "reference", "metric": "train ratings/sec", "value": val, "unit": "ratings/s", "n_gpus": args.gpus,
        "steps": n, "warmup": warm, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(name, w),
        "cpu_baseline": {"value": val, "unit": "ratings/s", "cores": cores, "kind": "port",
                         "sample": "%d full train steps of the workload (batch %d) by oracle/tfr_oracle.c, OpenMP on %d "
                                   "host threads; TensorFlow itself is absent" % (n, w["B"], cores)},
        "e2e": {"value": val, "unit": "ratings/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


# ---------------------------------------------------------------------------------------------------------------
def time_stream_steps(eng, steps, torch):
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    ev0.record()
    bufs = eng.run_stream_steps(steps, use_graph=True)
    ev1.record()
    torch.cuda.synchronize()
    return ev0.elapsed_time(ev1) / 1e3, bufs


DUMP_ROWS = 4096


def dump_rows(n):
    """The table rows --dump-outputs writes of a table of n rows: a fixed sample, ascending."""
    return np.sort(np.random.default_rng(0).choice(n, size=min(n, DUMP_ROWS), replace=False))


def last_step_outputs(eng, bufs, torch):
    """What the last timed step computed, as host arrays: the predictions run_stream_steps hands back (logits, infer:
    from the PRE-update tables) and the tables that step left behind, which alone show its update -- of users and items
    the rows dump_rows picks, since the ML-25M tables alone are 116 MB."""
    out = {k: bufs[k].cpu().numpy() for k in ("logits", "infer")}
    out["mu"] = eng.t["mu"].cpu().numpy()
    for side, n in (("user", eng.U), ("item", eng.I)):
        idx = torch.from_numpy(dump_rows(n)).to(eng.device)
        for tab in (side + "_bias", side + "_feat"):
            out[tab] = eng.t[tab][idx].cpu().numpy()
    return out


def write_outputs(outputs, out_dir):
    os.makedirs(out_dir, exist_ok=True)
    for name, a in outputs.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float32))


def _adam_tables(eng, ws, _lib):
    T, S = eng.t, eng.slots
    arr = (_lib.AdamTable * 4)()
    for k, (tab, rows, width, slot, gsum) in enumerate((("user_feat", eng.U, eng.d, eng.user_slot, ws.gsum_uf),
                                                        ("item_feat", eng.I, eng.d, eng.item_slot, ws.gsum_if),
                                                        ("user_bias", eng.U, 1, eng.user_slot, ws.gsum_ub),
                                                        ("item_bias", eng.I, 1, eng.item_slot, ws.gsum_ib))):
        arr[k].var, arr[k].m, arr[k].v = T[tab].data_ptr(), S["m_" + tab].data_ptr(), S["v_" + tab].data_ptr()
        arr[k].rows, arr[k].width, arr[k].slot, arr[k].gsum = rows, width, slot.data_ptr(), gsum
        arr[k].stride = (eng.feat_stride if width > 1 else 0)
    return arr


def kernel_roofline(eng, w, cols, steps, torch, peak, peak_src):
    """Times the dominant kernel (adam_stream_multi_kernel: the whole-table TF-Adam pass, every row of all four
    tables in one launch) live and IN SITU: complete pipelined steps are issued on the streams (same kernels, same
    side-stream fork as the captured graph: the next batch's assemble + id sort run beside the pass) with CUDA events
    recorded on the launching stream right before and right after the pass.  Stream-ordered events add almost
    nothing; event-record NODES inside a captured graph measured ~20 us more for the same launch (node-to-node
    latency on both sides), so the eager issue is used for this one number."""
    B, d, U, I = w["B"], w["d"], w["U"], w["I"]
    pairs = []

    def hook(tag, slot, stream):
        if tag == "pass_begin":
            pairs.append([torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)])
            pairs[-1][0].record(stream)
        else:
            pairs[-1][1].record(stream)
    eng.set_batch_cursor(0)
    eng.run_stream_steps(2, use_graph=True)   # leaves a buffer set primed for the batch at the cursor
    torch.cuda.synchronize()
    eng.timing_hook = hook
    try:
        # the steps are issued eagerly (one host call per kernel): park the device behind a spin kernel first so that
        # the host has queued every step before the first one runs -- the events then see device time only, never a
        # launch the host had not issued yet
        torch.cuda._sleep(int(3e7))
        eng.run_stream_steps(max(steps, 4), use_graph=False)
    finally:
        eng.timing_hook = None
    torch.cuda.synchronize()
    times = [p[0].elapsed_time(p[1]) for p in pairs[2:]]
    tot_ms, n = float(sum(times)), len(times)
    bytes_launch = 24.0 * (U + I) * (d + 1)
    achieved = bytes_launch / (tot_ms / n / 1e3) / 1e9
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "r02_pass_traffic.json")
    if not os.path.exists(tpath):
        tpath = os.path.join(ROOT, "profiles", "r01_pass_traffic.json")
    if os.path.exists(tpath):
        tj = json.load(open(tpath))
        if tj.get("workload") == w.get("name", "ml25m_d128_b65536"):
            traffic, traffic_src = tj["dram_bytes_per_launch"], "committed capture, not measured in this run: " + tj["source"]
    return {"bound": "hbm", "kernel": "adam_stream_multi_kernel (TF-Adam pass over every row of all tables, one launch)",
            "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src,
            "bytes_per_launch": bytes_launch, "launch_ms": tot_ms / n, "launches_timed": n,
            "how": "CUDA events on the launching stream right before / after the launch, inside complete pipelined "
                   "steps (in situ: the next batch's assemble + id sort run beside it on the side stream); all steps "
                   "are queued behind a spin kernel first, so the interval holds no host launch latency",
            "algorithmic_bytes": "24 B/param x (users+items) x (dim+1)", "traffic": traffic, "traffic_source": traffic_src}


def _n_partials(d, B):
    lanes = 1
    units = d // 4 if d % 4 == 0 else d
    while lanes < units and lanes < 32:
        lanes <<= 1
    rows_per_cta = 256 // lanes * 4
    return max(1, min(1024, (B + rows_per_cta - 1) // rows_per_cta))


def run_workload(name, args, torch, with_e2e=True, with_roofline=True, sample_clocks=True, dump=False):
    from tf_recomm_b200.engine import SvdEngine
    w = WORKLOADS[name]
    B = w["B"]
    cols = make_columns(w)
    np.random.seed(13575)  # svd_train_val.py:15 -- the reference's index stream
    eng = SvdEngine(w["U"], w["I"], w["d"], LR, REG, device_init_seed=13575)
    eng.set_train_data(*cols)
    n_train = len(cols[0])
    total = args.warmup + args.steps
    idx = np.concatenate([np.random.randint(0, n_train, (B,)) for _ in range(total)])
    eng.set_index_stream(idx, B)
    eng.run_stream_steps(args.warmup, use_graph=True)
    eng.prepare_stream_graphs(args.steps)   # capture + instantiate outside the timed region
    torch.cuda.synchronize()
    sampler = ClockSampler(torch.cuda.current_device()) if sample_clocks else None
    if sampler:
        sampler.start()
        time.sleep(0.3)
    secs, last = time_stream_steps(eng, args.steps, torch)
    # taken before anything below steps the engine again (the clock sampler's run-on lasts a wall-clock time)
    outputs = last_step_outputs(eng, last, torch) if dump else None
    if sampler and secs < 1.0:
        # keep the same work running long enough for the 100 ms clock sampler to see it under load
        eng.set_batch_cursor(0)
        t_end = time.time() + 1.5
        while time.time() < t_end:
            eng.set_batch_cursor(0)
            eng.run_stream_steps(min(total, 50), use_graph=True)
            torch.cuda.synchronize()
    clocks = sampler.stop() if sampler else None
    ms_step = secs / args.steps * 1e3
    value = B * args.steps / secs
    bytes_step = algorithmic_bytes_step(w["U"], w["I"], w["d"], B)
    peak, peak_src = measured_peaks()
    res = dict(value=value, ms_per_step=ms_step, bytes_step=bytes_step, hbm_gbs_step=bytes_step / (ms_step / 1e3) / 1e9,
               peak=peak, peak_src=peak_src, clocks=clocks, w=w, steps_per_epoch=n_train // B, outputs=outputs)
    if with_e2e:
        AHEAD, WARM = 3, 15
        rng = np.random.default_rng(3)
        drawn = []
        for _ in range(WARM + min(args.steps, 200)):   # at most 200 distinct timed batches (1.5 MB of host columns each)
            rows = rng.integers(0, n_train, B)
            drawn.append((cols[0][rows].astype(np.float64), cols[1][rows].astype(np.float64),
                          cols[2][rows].astype(np.float64)))   # float64 columns: what ShuffleIterator yields
        timed = [drawn[WARM + j % (len(drawn) - WARM)] for j in range(args.steps)]
        # the driver's loop (svd_train_val.py): batches t+1 .. t+3 have been handed over when step t is asked for and
        # returns its predictions (host) -- the later ones are being packed by the feed worker thread while t+1 is fetched
        # and its ids sorted under step t's table pass.  Every step's H2D (12 B / rating) and D2H (4 or 8 B / rating) are inside
        # the timed region, and so is the pipeline's fill: at small --steps it weighs on the number.

        def feed_loop(bs):
            for j in range(min(AHEAD, len(bs))):
                eng.prefetch_host(*bs[j])
            for j in range(len(bs)):
                if j + AHEAD < len(bs):
                    eng.prefetch_host(*bs[j + AHEAD])   # handed over before step j is asked for
                eng.train_step_host(*bs[j])
        # every step graph captured up front, then a warm-up in the same pattern (staging sets, pinned buffers, worker)
        eng.prepare_feed_graphs(B)
        feed_loop(drawn[:WARM])
        torch.cuda.synchronize()
        t0 = time.perf_counter()   # (the priming hand-overs are inside: every timed step's H2D is counted)
        feed_loop(timed)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        n = len(timed)
        res["e2e"] = {"value": B * n / dt, "unit": "ratings/s", "h2d_bytes_per_step": eng.h2d_bytes(B),
                      "d2h_bytes_per_step": eng.d2h_bytes(B), "ms_per_step": dt / n * 1e3, "steps": n,
                      "path": "SvdEngine.train_step_host + prefetch_host three batches ahead (what Session.run([train_op, logits, "
                              "infer], feed_dict) / Session.prefetch call; the loop of svd_train_val.py)"}
    if with_roofline and w["d"] % 4 == 0:
        res["roofline"] = kernel_roofline(eng, w, cols, min(args.steps, 20), torch, peak, peak_src)
    del eng
    torch.cuda.empty_cache()
    return res


def _claim_stdout():
    """The driver reads ONE JSON line from stdout.  Libraries write there too (NCCL prints its version banner to
    stdout): point file descriptor 1 at stderr for the whole run and keep the real stdout for the JSON line."""
    sys.stdout.flush()
    real = os.dup(1)
    os.dup2(2, 1)
    return os.fdopen(real, "w")


JSON_OUT = None


def emit(line):
    out = JSON_OUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    global JSON_OUT
    sys.dont_write_bytecode = True   # the benchmark writes nothing into the tree (which may be read-only), bytecode included
    JSON_OUT = _claim_stdout()
    sys.modules.setdefault("bench", sys.modules[__name__])  # bench_sharded / tools `import bench`: this very module
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps of value and e2e (default 200)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", type=str, default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", type=str, default=None)
    ap.add_argument("--no-also", action="store_true", help="skip the secondary ML-1M measurement")
    ap.add_argument("--cpu-steps", type=int, default=None, help="steps of the bounded CPU baseline sample")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (one GPU, --impl ours)")
    args = ap.parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    if args.dump_outputs and (args.gpus > 1 or world > 1 or args.impl != "ours"):
        ap.error("--dump-outputs needs a one-GPU run of --impl ours")
    if args.gpus > 1 or world > 1:
        import bench_sharded as sharded_bench
        return sharded_bench.main(args)
    name = args.workload or "ml25m_d128_b65536"
    w = WORKLOADS[name]
    if args.impl == "reference":
        if args.steps is None:
            args.steps = 10
        args.steps = min(args.steps, 40)   # bounded sample: ~37 ms per CPU step at the ML-25M shape
        if rank == 0:
            reference_arm(args, w, name)
        return
    if args.steps is None:
        args.steps = 200
    args.warmup = max(args.warmup, 3)
    import torch
    import tf_recomm_b200  # noqa: F401
    assert torch.cuda.is_available(), "bench.py needs a CUDA device; there is no CPU fallback (use --impl reference)"
    torch.cuda.set_device(0)
    r = run_workload(name, args, torch, dump=bool(args.dump_outputs))
    if args.dump_outputs:
        write_outputs(r["outputs"], args.dump_outputs)
    cores = os.cpu_count()
    cpu_steps = args.cpu_steps or (6 if w["d"] >= 64 else 60)
    tot, n = cpu_reference_run(w, cpu_steps, 2)
    cpu = {"value": w["B"] * n / tot, "unit": "ratings/s", "cores": cores, "kind": "port", "ms_per_step": tot / n * 1e3,
           "sample": "%d full train steps of the same workload (batch %d) by the CPU restatement of the TF path "
                     "(oracle/tfr_oracle.c, OpenMP, %d host threads); TensorFlow itself is absent" % (n, w["B"], cores)}
    steps_epoch = r["steps_per_epoch"]
    line = {
        "metric": "train ratings/sec", "value": r["value"], "unit": "ratings/s", "n_gpus": 1, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": (r["value"] / PUBLISHED_RATINGS_PER_S[name]) if name in PUBLISHED_RATINGS_PER_S else None,
        "dtype": "f32", "data": "synthetic",
        "config": workload_config(name, w),
        "notes": { "scaling_note": "--gpus N >= 2 measures BASELINE configs[4] (100M x 10M row-sharded: 170 GB of state "
                                   "that no single GPU holds), a different workload from this one: compare the multi-GPU "
                                   "lines with each other (baseline n_gpus = 2), not with this line",
                   "timing": "CUDA events around K replays of the captured step graph (each replay also assembles and "
                             "sorts the NEXT batch on a side stream: 6 kernels per step -- assemble, cursor advance, id sort, forward+segment sums, fix-up, Adam pass whose last CTA ends the step)"},
        "hbm": {"algorithmic_bytes_per_step": r["bytes_step"], "achieved_gbs": r["hbm_gbs_step"],
                "frac_of_measured_peak": r["hbm_gbs_step"] / r["peak"], "frac_of_nominal_8000": r["hbm_gbs_step"] / 8000.0,
                "peak_gbs": r["peak"], "peak_source": r["peak_src"]},
        "epoch_s": steps_epoch * r["ms_per_step"] / 1e3,
        "roofline": r.get("roofline"), "cpu_baseline": cpu, "e2e": r.get("e2e"), "clocks": r["clocks"],
        # our kernels launched inside the timed region: per step batch_assemble, advance_prefetch_cursor, dedup_sort,
        # segsum_tiles, segsum_fixup, adam_stream_multi (the graphs are captured before; counted from the step's structure)
        "gpu_launches": 6 * args.steps,
    }
    if not args.no_also and name == "ml25m_d128_b65536":
        a2 = argparse.Namespace(**vars(args))
        a2.steps, a2.warmup = 900, 20
        ra = run_workload("ml1m_d15_b10000", a2, torch, with_roofline=False, sample_clocks=False)
        wa = WORKLOADS["ml1m_d15_b10000"]
        line["also"] = {"workload": "ml1m_d15_b10000", "baseline_config": wa["config"], "value": ra["value"],
                        "unit": "ratings/s", "ms_per_step": ra["ms_per_step"], "steps": a2.steps,
                        "epoch_s": ra["steps_per_epoch"] * ra["ms_per_step"] / 1e3,
                        "readme_epoch_s": README_EPOCH_S["ml1m_d15_b10000"],
                        "vs_baseline": ra["value"] / PUBLISHED_RATINGS_PER_S["ml1m_d15_b10000"],
                        "e2e": ra.get("e2e"), "note": "launch/L2-bound: 5.2 MB/step, HBM fraction not meaningful"}
        try:
            line["also_allpairs"] = run_allpairs_workload(torch)
        except Exception as exc:
            line["also_allpairs"] = {"workload": "allpairs_162541x62423_d128", "error": repr(exc)}
        try:
            line["also_fm"] = run_fm_workload(torch)
        except Exception as exc:  # the headline line must not be lost to the secondary workload
            line["also_fm"] = {"workload": "fm_ktm_d20_b10000", "error": repr(exc)}
    emit(line)


def run_allpairs_workload(torch):
    """BASELINE configs[3]'s second half: all-pairs scoring of the ML-25M shape (als3.py:112, 2.6 TFLOP; the 40.6 GB score
    matrix is never written -- every consumer lives in the tcgen05 GEMM's epilogue).  ms, TFLOP/s and the fraction of
    the tf32 tensor peak (half the measured bf16 cuBLAS peak: tf32 MMAs run at half the bf16 rate) per consumer."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import allpairs_bench
    w = WORKLOADS["ml25m_d128_b65536"]
    res = allpairs_bench.run(w["U"], w["I"], w["d"], simt=False, reps=4)
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    bf16 = json.load(open(p)).get("bf16_tflops") if os.path.exists(p) else 1590.0
    tf32_peak = bf16 / 2.0
    for v in res.values():
        v["frac_of_tf32_peak"] = v["tflops"] / tf32_peak
    return {"workload": "allpairs_162541x62423_d128", "baseline_config": "configs[3] (all-pairs GEMM eval scoring)",
            "flop": 2.0 * w["U"] * w["I"] * w["d"], "dtype": "tf32 operands, fp32 accumulate (float64 rescore for rankings)",
            "tf32_peak_tflops": tf32_peak, "tf32_peak_source": "MEASURED_PEAKS.json bf16_tflops / 2 (burst)",
            "consumers": res}


def run_fm_workload(torch, epochs=12, warm_epochs=2):
    """BASELINE configs[2]: fm.py's 2nd-order FM, dim 20, on synthetic one-hot user / item / skill features of the
    ASSISTments shape (346,860 events, 4,217 + 26,688 + 123 features; SURVEY 8d #3), mini-batches of 10,000 CSR rows in
    file order, each batch's step one replayed graph.  Events / s over whole epochs, CUDA events."""
    import pandas as pd
    from tf_recomm_b200 import ktm
    from tf_recomm_b200._lib import LOSS_SIGMOID_CE
    from tf_recomm_b200.fm_engine import FmEngine
    users, items, outcomes, q = ktm.make_ktm_events()
    df = pd.DataFrame(dict(user=users, item=items, outcome=outcomes, wins=0, fails=0))
    U, I = int(users.max()) + 1, q.shape[0]
    X = ktm.df_to_sparse(df, ["users", "items", "skills"], U, I, q)
    B = 10000
    eng = FmEngine(X.shape[1], 20, 1e-2, 3e-2, flags=LOSS_SIGMOID_CE)
    chunks = np.array_split(np.arange(X.shape[0]), int(np.ceil(X.shape[0] / B)))
    batches = [eng.upload_csr(X[c], outcomes[c]) for c in chunks]
    for _ in range(warm_epochs):
        eng.run_epoch(batches)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(epochs):
        eng.run_epoch(batches)
    e1.record()
    torch.cuda.synchronize()
    secs = e0.elapsed_time(e1) / 1e3
    n_steps = epochs * len(batches)
    return {"workload": "fm_ktm_d20_b10000", "baseline_config": "configs[2]", "events": int(X.shape[0]),
            "features": int(X.shape[1]), "nnz_per_row": float(X.nnz / X.shape[0]), "dim": 20, "batch": B,
            "value": X.shape[0] * epochs / secs, "unit": "events/s", "ms_per_step": secs / n_steps * 1e3,
            "epoch_s": secs / epochs, "steps": n_steps,
            "model": "sigmoid cross-entropy + L2 + TF-Adam on (w0, W, V); libFM's MCMC (fm.py:104-110) is out of scope",
            "note": "launch/L2-bound: 15.6 MB of tables"}


if __name__ == "__main__":
    main()
