"""bench.py's output contract, checked on the arm that needs no GPU (--impl reference = the CPU restatement timed on the
host cores): exactly ONE JSON line on stdout, with the keys the driver reads.  On the GPU: --dump-outputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(argv):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + argv, cwd=ROOT, stdout=subprocess.PIPE,
                       stderr=subprocess.PIPE, timeout=600)
    assert p.returncode == 0, p.stderr.decode()[-2000:]
    lines = [l for l in p.stdout.decode().splitlines() if l.strip()]
    assert len(lines) == 1, lines
    return json.loads(lines[0])


def _run(extra):
    return _bench(["--impl", "reference", "--steps", "2", "--warmup", "1"] + extra)


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    d = _run(["--workload", "ml1m_d15_b10000"])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
              "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "ratings/s" and d["higher_is_better"] is True
    assert d["config"]["workload"] == "ml1m_d15_b10000" and d["dtype"] == "f32" and d["data"] == "synthetic"
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["cpu_baseline"]["value"] == d["value"] > 0
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert abs(d["value"] - 10000 / (d["ms_per_step"] / 1e3)) < 1e-6 * d["value"]


def test_reference_arm_under_a_multi_gpu_launch_prints_on_rank_0_only():
    """--gpus N > 1: rank 0 alone runs and prints; the other ranks exit 0 without work (no GPU, no process group)."""
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                        "--steps", "1"], cwd=ROOT, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=120)
    assert p.returncode == 0 and p.stdout.decode().strip() == ""


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_step_and_repeat(tmp_path):
    """--dump-outputs DIR: float32 arrays, equal array for array between two runs with the same arguments; --steps is the
    step count of both timed legs.  The logits are those of the LAST timed step: recomputed on the host (README model:
    mu + b_u + b_i + <p_u, q_i>) from the tables a run one step shorter left behind, on that step's batch of bench.py's
    seeded index stream; and that step moved the tables."""
    import bench

    def dump(steps, tag):
        out = tmp_path / tag
        d = _bench(["--workload", "ml1m_d15_b1000", "--steps", str(steps), "--warmup", "3", "--no-also", "--dump-outputs",
                    str(out)])
        assert d["steps"] == d["e2e"]["steps"] == steps
        return {p.stem: np.load(str(p)) for p in out.glob("*.npy")}
    a, b, before = dump(7, "a"), dump(7, "b"), dump(6, "before")
    assert set(a) == {"logits", "infer", "mu", "user_bias", "item_bias", "user_feat", "item_feat"}
    assert a["logits"].shape == a["infer"].shape == (1000,)
    assert a["user_feat"].shape == (4096, 15) and a["item_feat"].shape == (3952, 15) and a["item_bias"].shape == (3952,)
    for name in a:
        assert a[name].dtype == np.float32 and np.isfinite(a[name]).all(), name
        assert np.array_equal(a[name], b[name]), name
    w = bench.WORKLOADS["ml1m_d15_b1000"]
    B = w["B"]
    users, items, _ = bench.make_columns(w)
    np.random.seed(13575)   # bench.py's index stream: batch k of a run is draw k; the last timed step is 3 + 7 - 1
    rows = np.concatenate([np.random.randint(0, len(users), (B,)) for _ in range(10)])[9 * B:]
    u, i = users[rows], items[rows]
    ur, ir = bench.dump_rows(w["U"]), bench.dump_rows(w["I"])
    pu, pi = np.minimum(np.searchsorted(ur, u), len(ur) - 1), np.minimum(np.searchsorted(ir, i), len(ir) - 1)
    seen = (ur[pu] == u) & (ir[pi] == i)
    assert seen.sum() >= 500
    t = {k: v.astype(np.float64) for k, v in before.items()}
    ref = t["mu"][0] + t["user_bias"][pu] + t["item_bias"][pi] + np.sum(t["user_feat"][pu] * t["item_feat"][pi], axis=1)
    np.testing.assert_allclose(a["logits"][seen], ref[seen], rtol=1e-5, atol=1e-6)
    assert np.array_equal(a["infer"], a["logits"])   # the README head is the identity
    for name in ("mu", "user_bias", "item_bias", "user_feat", "item_feat"):
        assert not np.array_equal(a[name], before[name]), name
