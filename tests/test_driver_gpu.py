"""The reference's entry point on the GPU: `python svd_train_val.py` (svd_train_val.py:201-207) end to end, in the two
ways this repo can run its step loop, and the checkpoint it leaves (svd_train_val.py:197-198, adaptive_test.py:40)."""
import io
import os
import re
from contextlib import redirect_stdout

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _run(argv):
    import svd_train_val
    buf = io.StringIO()
    with redirect_stdout(buf):
        svd_train_val.main(argv)
    return buf.getvalue()


def _errors(text):
    """(epoch, train rmse, val rmse) from the lines `  e TRAIN(size=../.., rmse=..) TEST(size=.., rmse=..) ..(s)`
    (the reference's third print format, svd_train_val.py:180)."""
    out = []
    for line in text.splitlines():
        m = re.match(r"^\s*(\d+) TRAIN\(size=\d+/\d+, rmse=([0-9.]+)\) TEST\(size=\d+, rmse=([0-9.]+)\)", line)
        if m:
            out.append((int(m.group(1)), float(m.group(2)), float(m.group(3))))
    return out


def test_driver_session_and_stream_modes_agree(tmp_path):
    """--mode session feeds every batch through sess.run(feed_dict) like the reference; --mode stream replays captured
    graphs on device-resident columns with the SAME index stream (np.random.seed(13575) + ShuffleIterator draws):
    the reported train / val errors must coincide, and the RMSE must fall."""
    common = ["--synthetic", "ml1m", "--ratings", "60000", "--epochs", "4", "--batch", "1000", "--dim", "15"]
    a = _errors(_run(common + ["--mode", "session", "--checkpoint", str(tmp_path / "a.ckpt"), "--logdir", str(tmp_path / "la")]))
    b = _errors(_run(common + ["--mode", "stream", "--checkpoint", str(tmp_path / "b.ckpt"), "--logdir", str(tmp_path / "lb")]))
    assert len(a) >= 4 and len(a) == len(b)
    for (ea, ta, va), (eb, tb, vb) in zip(a, b):
        assert ea == eb
        assert ta == pytest.approx(tb, rel=2e-6) and va == pytest.approx(vb, rel=2e-6)
    assert a[-1][2] < a[0][2]          # validation RMSE went down
    za, zb = np.load(str(tmp_path / "a.ckpt")), np.load(str(tmp_path / "b.ckpt"))
    for n in ("mu", "user_bias", "item_bias", "user_feat", "item_feat", "m_user_feat", "v_item_feat"):
        assert np.array_equal(za[n], zb[n]), n   # same kernels, same batches: bit-identical tables
    assert int(za["__step__"][0]) == int(zb["__step__"][0]) > 0


def test_checkpoint_restore_continues_bit_identically(tmp_path):
    """save -> restore into a fresh engine -> the next steps equal those of the engine that never stopped (interleaved
    tables, stamped slot maps and the Adam scalars all survive the round trip)."""
    from tf_recomm_b200 import init
    from tf_recomm_b200.engine import SvdEngine
    rng = np.random.default_rng(0)
    U, I, d, B = 300, 200, 128, 2048
    tabs = init.init_tables(U, I, d, seed=2)
    eng = SvdEngine(U, I, d, 1e-3, 0.05, tables=tabs)
    batches = [(rng.integers(0, U, B).astype(np.int32), rng.integers(0, I, B).astype(np.int32),
                rng.integers(1, 6, B).astype(np.float32)) for _ in range(6)]
    for b in batches[:3]:
        eng.train_step(*b)
    path = str(tmp_path / "fm.ckpt")
    eng.save(path)
    other = SvdEngine(U, I, d, 1e-3, 0.05, tables=init.init_tables(U, I, d, seed=9))
    other.restore(path)
    assert other.global_step == 3
    for b in batches[3:]:
        la, _ = eng.train_step(*b)
        lb, _ = other.train_step(*b)
        assert np.array_equal(la.cpu().numpy(), lb.cpu().numpy())
    ta, tb = eng.get_tables(), other.get_tables()
    for n in ta:
        assert np.array_equal(ta[n], tb[n]), n


def test_driver_fork_variant_reports_acc_auc_nll(tmp_path):
    """The code as written (ops.py:44,85-89,125,145: |q| in the dot, sigmoid cross-entropy, bias L2, SGD) through the
    reference's DISCRETE branch: accuracy / AUC / mean NLL per epoch (svd_train_val.py:94-98,138-143,156)."""
    text = _run(["--synthetic", "ml1m", "--ratings", "40000", "--epochs", "3", "--batch", "500", "--dim", "20",
                 "--variant", "fork", "--lr", "0.005", "--reg", "0.01", "--checkpoint", os.devnull,
                 "--logdir", str(tmp_path / "log")])
    rows = re.findall(r"^\s*(\d+) TRAIN\(size=\d+/\d+, macc=([0-9.]+), mauc=([0-9.]+), mnll=([0-9.]+)\) "
                      r"TEST\(size=\d+, macc=([0-9.]+), auc=([0-9.]+), mnll=([0-9.]+)\)", text, flags=re.M)
    assert len(rows) >= 3, text[-400:]
    first, last = rows[0], rows[-1]
    assert all(0.0 <= float(x) <= 1.0 for r in rows for x in (r[1], r[2], r[4], r[5]))
    assert float(last[6]) < float(first[6])     # validation NLL fell
    assert float(last[5]) > 0.5                 # validation AUC above chance


def test_driver_reads_the_reference_csv_layout(tmp_path, monkeypatch):
    """data/<name>/{train,val,test}.csv + config.yml (dataio.py:8-16,38-54): header-less user,item,outcome,wins,fails."""
    import yaml
    rng = np.random.default_rng(0)
    folder = tmp_path / "data" / "tiny"
    folder.mkdir(parents=True)
    U, I = 40, 30
    for name, n in (("train", 3000), ("val", 400), ("test", 400)):
        u, i = rng.integers(0, U, n), rng.integers(0, I, n)
        r = np.clip(np.rint(3.5 + 0.8 * np.sin(u) + 0.6 * np.cos(i) + rng.normal(0, 0.5, n)), 1, 5)
        with open(folder / (name + ".csv"), "w") as f:
            for k in range(n):
                f.write("%d,%d,%d,0,0\n" % (u[k], i[k], r[k]))
    with open(folder / "config.yml", "w") as f:
        yaml.safe_dump(dict(USER_NUM=U, ITEM_NUM=I, NB_CLASSES=5, BATCH_SIZE=100), f)
    monkeypatch.chdir(tmp_path)
    rows = _errors(_run(["--dataset", "tiny", "--epochs", "5", "--batch", "100", "--dim", "8", "--lr", "0.01",
                         "--checkpoint", str(tmp_path / "fm.ckpt"), "--logdir", str(tmp_path / "log")]))
    assert len(rows) >= 5 and rows[-1][2] < rows[0][2]
    z = np.load(str(tmp_path / "fm.ckpt"))
    assert z["user_feat"].shape == (U, 8) and z["item_feat"].shape == (I, 8)


def test_driver_fork_device_metrics_equal_host_metrics_and_tensorboard(tmp_path):
    """DISCRETE branch: ACC / AUC / NLL computed on the device (tfr_binary_metrics) print the same lines as the reference's
    host code (numpy sigmoid / round, sklearn-equivalent AUC); and the two runs leave the reference's TensorBoard scalars
    `training_error` / `test_error` (svd_train_val.py:20-21,57,189-192) in an event file."""
    from tf_recomm_b200 import summary
    common = ["--synthetic", "ml1m", "--ratings", "30000", "--epochs", "2", "--batch", "500", "--dim", "20",
              "--variant", "fork", "--lr", "0.005", "--reg", "0.01", "--checkpoint", os.devnull]
    pat = (r"^\s*(\d+) TRAIN\(size=\d+/\d+, macc=([0-9.]+), mauc=([0-9.]+), mnll=([0-9.]+)\) "
           r"TEST\(size=\d+, macc=([0-9.]+), auc=([0-9.]+), mnll=([0-9.]+)\)")
    dev = re.findall(pat, _run(common + ["--logdir", str(tmp_path / "tb")]), flags=re.M)
    host = re.findall(pat, _run(common + ["--logdir", "", "--host-metrics"]), flags=re.M)
    assert len(dev) == len(host) >= 2
    for a, b in zip(dev, host):
        assert a[0] == b[0]
        for x, y in zip(a[1:], b[1:]):
            assert float(x) == pytest.approx(float(y), abs=2e-6)
    files = list((tmp_path / "tb").iterdir())
    assert len(files) == 1 and files[0].name.startswith("events.out.tfevents.")
    ev = summary.read_events(str(files[0]))
    tags = {t for _, t, _ in ev}
    assert {"training_error", "test_error", "train_macc", "test_auc", "test_mnll"} <= tags
    assert [s for s, t, _ in ev if t == "test_auc"][0] == 0        # the first report comes after ONE step (:106)


def test_driver_readme_tensorboard_scalars(tmp_path):
    from tf_recomm_b200 import summary
    text = _run(["--synthetic", "ml1m", "--ratings", "30000", "--epochs", "3", "--batch", "1000", "--dim", "15",
                 "--checkpoint", os.devnull, "--logdir", str(tmp_path / "log")])
    rows = _errors(text)
    ev = summary.read_events(str(next((tmp_path / "log").iterdir())))
    tr = [(s, v) for s, t, v in ev if t == "training_error"]
    te = [(s, v) for s, t, v in ev if t == "test_error"]
    assert len(tr) == len(te) == len(rows)
    nb = 27000 // 1000
    for (e, a, b), (s1, v1), (s2, v2) in zip(rows, tr, te):
        assert s1 == s2 == e * nb                                   # add_summary(summary, i), i = the step index
        assert v1 == pytest.approx(a, abs=2e-6) and v2 == pytest.approx(b, abs=2e-6)
