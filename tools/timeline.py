"""Per-kernel start/end times inside ONE graph-replayed train step, from in-kernel %globaltimer stamps
(tfr_opt_set_timeline).  Usage (GPU box): python tools/timeline.py [workload] [overlap 0..3]
TFR_TL_STEPS=2: one PAIR of steps per record (two steps per table pass): the slots of the forward / segment-sum kernels
then span both steps' launches."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
import tf_recomm_b200  # noqa: E402,F401
from tf_recomm_b200.engine import SvdEngine  # noqa: E402


def main():
    name = sys.argv[1] if len(sys.argv) > 1 else "ml25m_d128_b65536"
    overlap = int(sys.argv[2]) if len(sys.argv) > 2 else 3
    use_graph = (sys.argv[3] != "eager") if len(sys.argv) > 3 else True
    pipeline = (sys.argv[4] == "pipe") if len(sys.argv) > 4 else True
    w = bench.WORKLOADS[name]
    cols = bench.make_columns(w)
    eng = SvdEngine(w["U"], w["I"], w["d"], bench.LR, bench.REG, device_init_seed=1)
    eng.overlap = overlap
    if os.environ.get("TFR_PREFETCH_AT_START"):
        eng.prefetch_at_start = int(os.environ["TFR_PREFETCH_AT_START"])
    if os.environ.get("TFR_GRAPH_STEPS"):
        eng.graph_steps = int(os.environ["TFR_GRAPH_STEPS"])
    eng.set_train_data(*cols)
    B, reps = w["B"], 12
    per = int(os.environ.get("TFR_TL_STEPS", "1"))
    np.random.seed(1)
    eng.set_index_stream(np.random.randint(0, len(cols[0]), (per * reps + 8) * B), B)
    eng.enable_timeline()
    eng.run_stream_steps(8, use_graph=use_graph, pipeline=pipeline)
    torch.cuda.synchronize()
    acc = {}
    for _ in range(reps):
        eng.reset_timeline()
        torch.cuda.synchronize()
        eng.run_stream_steps(per, use_graph=use_graph, pipeline=pipeline)
        torch.cuda.synchronize()
        for k, (a, b) in eng.read_timeline().items():
            acc.setdefault(k, []).append((a, b))
    print("workload %s overlap=%d  (us from the first kernel entry of %d step(s); median of %d records)"
          % (name, overlap, per, reps))
    end_all = 0
    for k in eng.TL_NAMES:
        if k in acc:
            a = np.median([x[0] for x in acc[k]]); b = np.median([x[1] for x in acc[k]])
            end_all = max(end_all, b)
            print("%-18s start %8.1f  end %8.1f  dur %8.1f" % (k, a, b, b - a))
    print("step span %.1f us" % end_all)
    eng.set_batch_cursor(0)
    eng.run_stream_steps(1, use_graph=use_graph, pipeline=pipeline)
    import time
    torch.cuda.synchronize(); t0 = time.perf_counter()
    nb = 64
    eng.set_index_stream(np.random.randint(0, len(cols[0]), (nb + 8) * B), B)
    eng.run_stream_steps(nb, use_graph=use_graph, pipeline=pipeline)
    eng.set_batch_cursor(0)
    torch.cuda.synchronize(); t0 = time.perf_counter()
    eng.run_stream_steps(nb, use_graph=use_graph, pipeline=pipeline)
    torch.cuda.synchronize()
    print("back-to-back: %.1f us/step (%s)" % ((time.perf_counter() - t0) / nb * 1e6, "graph" if use_graph else "eager"))


if __name__ == "__main__":
    main()
