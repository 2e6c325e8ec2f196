"""Train + validate the matrix-factorization model: the reference's entry point (svd_train_val.py in
jilljenn/TF-recomm), with the TensorFlow graph replaced by tf-recomm_b200's CUDA path.

    python svd_train_val.py --synthetic ml1m --epochs 100 --batch 1000            # README run shape
    python svd_train_val.py --dataset mydata --variant fork                          # data/<name>/{train,val,test}.csv

Same protocol as the reference's svd() (file:line into /root/reference/svd_train_val.py): nb_batches = len(train)
// BATCH_SIZE steps per "epoch" (:24), batches drawn with replacement by ShuffleIterator under np.random.seed(13575)
(:15,:26), predictions fetched from the pre-update tables (:70-72), trailing window of the last nb_batches batches for
the train error (:59-64,:104-108), whole validation set in one forward batch (:33-38,:120-122), first report after ONE
step (:106, i % nb_batches == 0 at i = 0), the reference's three print formats (:156,:170,:180) and a checkpoint at the
end (:197-198).  What the reference left undefined (BATCH_SIZE, USER_NUM, ITEM_NUM, NB_CLASSES, the DATASET_NAME
argument, cost_l2/rates/pred_batch on the non-DISCRETE branch -- SURVEY Appendix B) is defined here.

Two ways to run the step loop:
  --mode session   (default) the reference's loop verbatim: next(iter_train) -> sess.run(feed_dict) per step.
  --mode stream    the same batches, but the training columns live in HBM and the whole epoch's index stream is
                   drawn up front (same RandomState consumption); each step is one replay of a captured CUDA graph.

--solver als trains by alternating least squares instead (SvdEngine.als_sweep): every epoch is one sweep that solves each
user row, then each item row, exactly in float64 against the other side, then updates mu; TRAIN is the RMSE over the whole
training set after the sweep.  --batch, --lr and --mode do not apply to it.

--solver ials trains the same tables from implicit feedback instead (SvdEngine.ials_sweep, Hu, Koren and Volinsky 2008):
every training pair is an interaction of weight 1 (duplicates add), confidence 1 + --alpha * weight, every other pair a
0 of confidence 1, --reg the lambda of lambda * I.  Every epoch is one sweep; the IMPLICIT line is the loss over all user x
item pairs after it.  Biases and mu are 0 after a sweep, so the model ranks by p_u . q_i.  --topk is required (RMSE against
ratings means nothing for this model); --batch, --lr and --mode do not apply.

--topk K adds, after every report, the top-K recommendation quality on the validation split: each user is ranked over
the items they did not rate in training, and hit rate / precision / recall / NDCG at K are measured against their
validation items (rated >= --topk-min-rating; on the DISCRETE branch, an outcome of 1).
"""
import argparse
import contextlib
import os
import time
from collections import deque

import numpy as np

import tf_recomm_b200  # noqa: F401
from tf_recomm_b200 import config, dataio, ops, summary, synthetic


def roc_auc(y_true, score):
    """Area under the ROC curve by the rank statistic (ties averaged) -- what sklearn.metrics.roc_auc_score,
    used at svd_train_val.py:97,141, computes."""
    y = np.asarray(y_true) > 0.5
    n_pos, n_neg = int(y.sum()), int((~y).sum())
    if n_pos == 0 or n_neg == 0:
        return float("nan")
    from scipy.stats import rankdata
    r = rankdata(score)
    return float((r[y].sum() - n_pos * (n_pos + 1) / 2.0) / (n_pos * n_neg))


def _graph(args):
    """The reference's graph (:30-56): -> ((user, item, rate, wins, fails) placeholders, infer, logits, cost, train_op)."""
    user_batch = ops.placeholder(ops.int32, shape=[None], name="id_user")
    item_batch = ops.placeholder(ops.int32, shape=[None], name="id_item")
    rate_batch = ops.placeholder(ops.float32, shape=[None])
    wins_batch = ops.placeholder(ops.float32, shape=[None], name="nb_wins")
    fails_batch = ops.placeholder(ops.float32, shape=[None], name="nb_fails")
    ops.reset_default_graph()
    infer, logits, regularizer, _, _, _, _ = ops.inference_svd(
        user_batch, item_batch, wins_batch, fails_batch, user_num=args.user_num, item_num=args.item_num, dim=args.dim,
        device=config.DEVICE, variant=args.variant)
    ops.train.get_or_create_global_step()
    cost, train_op = ops.optimization(infer, logits, regularizer, rate_batch, learning_rate=args.lr, reg=args.reg,
                                      device=config.DEVICE)
    return (user_batch, item_batch, rate_batch, wins_batch, fails_batch), infer, logits, cost, train_op


@contextlib.contextmanager
def _session(args, log):
    """The reference's graph in an initialised session (:30-57): -> (sess, engine, writer, _graph's tuple), writer the
    TensorBoard FileWriter or None.  When the training loop is done: the writer closed and the checkpoint (:197-198)."""
    graph = _graph(args)
    init_op = ops.group(ops.global_variables_initializer(), ops.local_variables_initializer())
    saver = ops.train.Saver()
    with ops.Session() as sess:
        sess.run(init_op)
        writer = summary.FileWriter(args.logdir) if getattr(args, "logdir", None) else None   # :57
        yield sess, ops.session.current_model().engine, writer, graph
        if writer is not None:
            writer.close()
        if args.checkpoint:
            path = os.path.join(config.BASE_DIR, args.checkpoint)
            log(path)
            saver.save(sess, path)


def _topk(engine, k, test, min_rating, exclude, rec, log):
    """A report's TOPK line: top-k quality on the validation split (SvdEngine.ranking_metrics), kept in rec["topk"].
    -> the seconds it took, which the next report's elapsed time leaves out."""
    t_topk = time.time()
    rm = engine.ranking_metrics(k, test["user"], test["item"], rates=test["outcome"], min_rating=min_rating,
                                exclude=exclude)
    rec["topk"] = rm
    log("TOPK(k={:d}, users={:d}, hr={:f}, precision={:f}, recall={:f}, ndcg={:f})".format(
        k, rm["n_users"], rm["hr"], rm["precision"], rm["recall"], rm["ndcg"]))
    return time.time() - t_topk


def _topk_summaries(writer, rm, step):
    for tag, key in (("hr_at_k", "hr"), ("precision_at_k", "precision"), ("recall_at_k", "recall"), ("ndcg_at_k", "ndcg")):
        writer.add_summary(summary.make_scalar_summary(tag, rm[key]), step)


def svd(train, test, args, log=print):
    BATCH_SIZE = args.batch
    nb_batches = len(train["user"]) // BATCH_SIZE
    discrete = args.variant == "fork"
    host_metrics = bool(getattr(args, "host_metrics", False))
    cols = ["user", "item", "outcome", "wins", "fails"]
    iter_train = dataio.ShuffleIterator([train[c] for c in cols], batch_size=BATCH_SIZE)
    iter_test = dataio.OneEpochIterator([test[c] for c in cols], batch_size=-1)
    history = []
    with _session(args, log) as (sess, engine, writer, graph):
        (user_batch, item_batch, rate_batch, wins_batch, fails_batch), infer, logits, cost, train_op = graph
        log("{} {} {} {}".format("epoch", "train_error", "val_error", "elapsed_time"))
        train_se = deque(maxlen=nb_batches)
        train_nll = deque(maxlen=nb_batches)
        train_acc = deque(maxlen=nb_batches)
        train_auc = deque(maxlen=nb_batches)
        if args.mode == "stream":
            engine.set_train_data(train["user"], train["item"], train["outcome"])
            engine.set_se_ring(nb_batches)
        topk = int(getattr(args, "topk", 0) or 0)
        if topk:
            # the training pairs are never recommended: their CSR is built once, not per report
            topk_exclude = engine.pair_csr(train["user"], train["item"])
            topk_min_rating = 1.0 if discrete else float(args.topk_min_rating)
        start = time.time()
        total_steps = args.epochs * nb_batches
        i = 0

        def feed_of(b):
            return {user_batch: b[0], item_batch: b[1], rate_batch: b[2], wins_batch: b[3], fails_batch: b[4]}
        # session mode: this driver owns the iterator, so batches i+1 .. i+3 are drawn (same RandomState order as the
        # reference's loop: one draw per step, total_steps draws in all) and handed to sess.prefetch BEFORE step i is
        # asked for -- the later ones are being packed by the feed worker while i+1 is fetched and sorted under step i's pass
        AHEAD = 3
        drawn = []          # batches handed over, not stepped yet
        n_drawn = 0

        def draw_ahead():
            nonlocal n_drawn
            while len(drawn) < AHEAD + 1 and n_drawn < total_steps:
                drawn.append(next(iter_train))
                n_drawn += 1
                sess.prefetch(feed_of(drawn[-1]))
        if not (args.mode == "stream" and not discrete):
            draw_ahead()
        while i < total_steps:
            if args.mode == "stream" and not discrete:
                # steps i .. next report: the first report comes after one step, then every nb_batches
                n = 1 if i == 0 else min(nb_batches, total_steps - i)
                engine.set_index_stream(iter_train.draw_index_stream(n), BATCH_SIZE)
                engine.run_stream_steps(n, use_graph=True)
                i += n
                ring = engine.se_ring.cpu().numpy()
                filled = min(i, nb_batches)
                train_rmse = float(np.sqrt(ring[:filled].sum() / (filled * BATCH_SIZE)))
                report_at = i - 1
                last_batch = BATCH_SIZE
                if report_at % nb_batches != 0:
                    continue  # the tail after the last full epoch is trained but not reported (:106)
            else:
                draw_ahead()
                cur = drawn.pop(0)
                train_users, train_items, train_rates, train_wins, train_fails = cur
                _, train_logits, train_infer = sess.run([train_op, logits, infer], feed_dict=feed_of(cur))
                if discrete:
                    if host_metrics:   # the reference's own host code (:94-98), kept as the cross-check
                        nll_batch = sess.run(cost, feed_dict={rate_batch: train_rates, logits: train_logits})
                        proba_batch = ops.sigmoid(train_logits)
                        train_acc.append(np.mean(np.round(proba_batch) == train_rates))
                        train_auc.append(roc_auc(train_rates, proba_batch))
                        train_nll.append(nll_batch)
                    else:                   # same three numbers from the step's device-resident logits and ratings
                        mt = engine.last_step_metrics(len(train_users))
                        train_acc.append(mt["n_correct"] / mt["n"])
                        train_auc.append(mt["auc"])
                        train_nll.append(mt["nll_sum"])
                else:
                    train_se.append(np.power(train_rates - train_infer, 2))
                report_at = i
                i += 1
                last_batch = len(train_users)
                if report_at % nb_batches != 0:
                    continue
                train_rmse = float(np.sqrt(np.mean(train_se))) if train_se else float("nan")
            # ---- report (svd_train_val.py:106-193) ----
            test_se, test_acc, test_nll, test_auc = [], [], [], 0.0
            for test_users, test_items, test_rates, test_wins, test_fails in iter_test:
                if discrete and not host_metrics:
                    # forward + ACC / AUC / NLL without the logits ever leaving the device (32 bytes come back)
                    lg_dev, _ = engine.forward(test_users, test_items)
                    mt = engine.binary_metrics(lg_dev, test_rates)
                    test_acc.append(mt["n_correct"] / mt["n"])
                    test_auc = mt["auc"]
                    test_nll.append(mt["nll_sum"])
                    continue
                test_logits, test_infer = sess.run([logits, infer], feed_dict={
                    user_batch: test_users, item_batch: test_items, wins_batch: test_wins, fails_batch: test_fails})
                if discrete:
                    nll_batch = sess.run(cost, feed_dict={rate_batch: test_rates, logits: test_logits})
                    proba_batch = ops.sigmoid(test_logits)
                    test_acc.append(np.mean(np.round(proba_batch) == test_rates))
                    test_auc = roc_auc(test_rates, proba_batch)
                    test_nll.append(nll_batch)
                else:
                    test_se.append(np.power(test_rates - test_infer, 2))
            end = time.time()
            epoch = report_at // nb_batches
            if discrete:
                rec = dict(epoch=epoch, train_macc=float(np.mean(train_acc)), train_mauc=float(np.mean(train_auc)),
                           train_mnll=float(np.mean(train_nll) / BATCH_SIZE), test_macc=float(np.mean(test_acc)),
                           test_auc=float(test_auc), test_mnll=float(np.mean(test_nll) / len(test["user"])),
                           elapsed=end - start)
                log("{:3d} TRAIN(size={:d}/{:d}, macc={:f}, mauc={:f}, mnll={:f}) TEST(size={:d}, macc={:f}, auc={:f}, "
                    "mnll={:f}) {:f}(s)".format(epoch, last_batch, len(train["user"]), rec["train_macc"],
                                                rec["train_mauc"], rec["train_mnll"], len(test["user"]),
                                                rec["test_macc"], rec["test_auc"], rec["test_mnll"], end - start))
            else:
                test_rmse = float(np.sqrt(np.mean(test_se)))
                rec = dict(epoch=epoch, train_rmse=train_rmse, test_rmse=test_rmse, elapsed=end - start)
                log("{:3d} TRAIN(size={:d}/{:d}, rmse={:f}) TEST(size={:d}, rmse={:f}) {:f}(s)".format(
                    epoch, last_batch, len(train["user"]), train_rmse, len(test["user"]), test_rmse, end - start))
            if topk:
                end += _topk(engine, topk, test, topk_min_rating, topk_exclude, rec, log)
            history.append(rec)
            if writer is not None:
                # svd_train_val.py:189-192: train_rmse / test_rmse under these two tags (NaN on the DISCRETE branch, where
                # the reference's train_se stays empty; the branch's own numbers go out under tags of their own)
                writer.add_summary(summary.make_scalar_summary("training_error", rec.get("train_rmse", float("nan"))), report_at)
                writer.add_summary(summary.make_scalar_summary("test_error", rec.get("test_rmse", float("nan"))), report_at)
                if discrete:
                    for tag in ("train_macc", "train_mauc", "train_mnll", "test_macc", "test_auc", "test_mnll"):
                        writer.add_summary(summary.make_scalar_summary(tag, rec[tag]), report_at)
                if topk:
                    _topk_summaries(writer, rec["topk"], report_at)
                writer.flush()
            start = end
    return history


def svd_als(train, test, args, log=print):
    """--solver als: the same model, initialisation, report lines, --topk, summaries and checkpoint as svd(), trained by one
    ALS sweep per epoch.  TRAIN(size=N/N) is the RMSE over every training rating (tfr_svd_objective), TEST the forward's."""
    history = []
    n_train, n_test = len(train["user"]), len(test["user"])
    with _session(args, log) as (sess, engine, writer, graph):
        (user_batch, item_batch, _, wins_batch, fails_batch), infer, logits, _, _ = graph
        data = engine.als_data(train["user"], train["item"], train["outcome"])
        topk = int(getattr(args, "topk", 0) or 0)
        if topk:
            topk_exclude = engine.pair_csr(train["user"], train["item"])
        log("{} {} {} {}".format("epoch", "train_error", "val_error", "elapsed_time"))
        start = time.time()
        for epoch in range(args.epochs):
            failed = engine.als_sweep(data, reg=args.reg)
            train_rmse = engine.training_objective(data, reg=args.reg)["rmse"]
            n_failed = int(failed.item())
            if n_failed:
                log("ALS: %d rows kept their previous values (a pivot was not > 0)" % n_failed)
            test_se = []
            for test_users, test_items, test_rates, test_wins, test_fails in dataio.OneEpochIterator(
                    [test[c] for c in ("user", "item", "outcome", "wins", "fails")], batch_size=-1):
                _, test_infer = sess.run([logits, infer], feed_dict={
                    user_batch: test_users, item_batch: test_items, wins_batch: test_wins, fails_batch: test_fails})
                test_se.append(np.power(test_rates - test_infer, 2))
            end = time.time()
            test_rmse = float(np.sqrt(np.mean(test_se)))
            rec = dict(epoch=epoch, train_rmse=train_rmse, test_rmse=test_rmse, elapsed=end - start)
            log("{:3d} TRAIN(size={:d}/{:d}, rmse={:f}) TEST(size={:d}, rmse={:f}) {:f}(s)".format(
                epoch, n_train, n_train, train_rmse, n_test, test_rmse, end - start))
            if topk:
                end += _topk(engine, topk, test, float(args.topk_min_rating), topk_exclude, rec, log)
            history.append(rec)
            if writer is not None:
                writer.add_summary(summary.make_scalar_summary("training_error", train_rmse), epoch)
                writer.add_summary(summary.make_scalar_summary("test_error", test_rmse), epoch)
                if topk:
                    _topk_summaries(writer, rec["topk"], epoch)
                writer.flush()
            start = end
    return history


def svd_ials(train, test, args, log=print):
    """--solver ials: the same model, initialisation, --topk lines, summaries and checkpoint as svd(), trained by one iALS
    sweep per epoch from the training pairs as implicit feedback.  IMPLICIT(...) is the loss after the sweep."""
    history = []
    with _session(args, log) as (sess, engine, writer, _):
        data = engine.ials_data(train["user"], train["item"])
        topk_exclude = engine.pair_csr(train["user"], train["item"])
        log("{} {} {}".format("epoch", "implicit_loss", "elapsed_time"))
        start = time.time()
        for epoch in range(args.epochs):
            failed = engine.ials_sweep(data, args.alpha, reg=args.reg)
            obj = engine.implicit_objective(data, args.alpha, reg=args.reg)
            n_failed = int(failed.item())
            if n_failed:
                log("iALS: %d rows kept their previous values (a pivot was not > 0)" % n_failed)
            end = time.time()
            rec = dict(epoch=epoch, implicit_loss=obj["loss"], elapsed=end - start)
            log("{:3d} IMPLICIT(pairs={:d}, loss={:.10g}, observed={:.10g}, all_pairs={:.10g}, penalty={:.10g}) {:f}(s)"
                .format(epoch, obj["n"], obj["loss"], obj["observed"], obj["all_pairs"], obj["penalty"], end - start))
            end += _topk(engine, args.topk, test, float(args.topk_min_rating), topk_exclude, rec, log)
            history.append(rec)
            if writer is not None:
                writer.add_summary(summary.make_scalar_summary("implicit_loss", obj["loss"]), epoch)
                _topk_summaries(writer, rec["topk"], epoch)
                writer.flush()
            start = end
    return history


def load(args):
    if args.dataset:
        df_train, df_val, df_test = dataio.get_data(args.dataset)
        folder, _, _, _, cfg_file, _ = dataio.build_paths(args.dataset)
        if os.path.exists(cfg_file):
            cfg = config.load_dataset_config(cfg_file)
            args.user_num = args.user_num or cfg.get("USER_NUM")
            args.item_num = args.item_num or cfg.get("ITEM_NUM")
        as_cols = lambda df: {c: df[c].to_numpy() for c in dataio.COLUMNS}  # noqa: E731
        train, val = as_cols(df_train), as_cols(df_val)
        print("Train", df_train.shape); print("Val", df_val.shape); print("Test", df_test.shape)
    else:
        U, I, N = synthetic.SHAPES[args.synthetic]
        if args.ratings:
            N = args.ratings
        users, items, rates = synthetic.make_ratings(U, I, N, seed=config.SEED, binary=(args.variant == "fork"))
        (tu, ti, tr), (vu, vi, vr) = synthetic.split(users, items, rates)
        z = lambda n: np.zeros(n, np.float32)  # noqa: E731
        train = dict(user=tu, item=ti, outcome=tr, wins=z(len(tu)), fails=z(len(tu)))
        val = dict(user=vu, item=vi, outcome=vr, wins=z(len(vu)), fails=z(len(vu)))
        args.user_num, args.item_num = args.user_num or U, args.item_num or I
        print("Train", (len(tu), 5)); print("Val", (len(vu), 5))
    args.user_num = args.user_num or int(max(train["user"].max(), val["user"].max())) + 1
    args.item_num = args.item_num or int(max(train["item"].max(), val["item"].max())) + 1
    return train, val


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--dataset", type=str, default=None, help="data/<name>/{train,val,test}.csv (dataio.get_data)")
    ap.add_argument("--synthetic", type=str, default="ml1m", choices=sorted(synthetic.SHAPES))
    ap.add_argument("--ratings", type=int, default=None, help="override the number of synthetic ratings")
    ap.add_argument("--variant", type=str, default=config.MODEL_VARIANT, choices=["readme", "fork"])
    ap.add_argument("--solver", type=str, default="adam", choices=["adam", "als", "ials"],
                    help="adam: the reference's optimizer steps (default); als: exact alternating least squares sweeps "
                         "on the device, README variant only, dim <= 128; ials: implicit-feedback ALS sweeps (the "
                         "training pairs as interactions), README variant only, dim <= 128, needs --topk")
    ap.add_argument("--alpha", type=float, default=1.0,
                    help="--solver ials: confidence 1 + alpha * weight of an interaction (>= 0)")
    ap.add_argument("--epochs", type=int, default=config.EPOCH_MAX, help="epochs (with --solver als: sweeps)")
    ap.add_argument("--batch", type=int, default=config.BATCH_SIZE, help="batch size (not used by --solver als)")
    ap.add_argument("--dim", type=int, default=config.DIM)
    ap.add_argument("--lr", type=float, default=config.LEARNING_RATE, help="learning rate (not used by --solver als)")
    ap.add_argument("--reg", type=float, default=config.LAMBDA_REG)
    ap.add_argument("--user-num", dest="user_num", type=int, default=None)
    ap.add_argument("--item-num", dest="item_num", type=int, default=None)
    ap.add_argument("--mode", type=str, default="session", choices=["session", "stream"],
                    help="step loop of --solver adam (not used by --solver als)")
    ap.add_argument("--checkpoint", type=str, default="fm.ckpt")
    ap.add_argument("--logdir", type=str, default="/tmp/svd/log",
                    help="TensorBoard event files (svd_train_val.py:57); empty string = none")
    ap.add_argument("--host-metrics", dest="host_metrics", action="store_true",
                    help="DISCRETE branch: ACC / AUC / NLL with the reference's host code instead of on the device")
    ap.add_argument("--topk", type=int, default=0,
                    help="after every report, hit rate / precision / recall / NDCG at this k on the validation split, "
                         "training items excluded from the ranking (0 = off)")
    ap.add_argument("--topk-min-rating", dest="topk_min_rating", type=float, default=4.0,
                    help="README variant: the validation ratings that count as relevant for --topk")
    args = ap.parse_args(argv)
    if args.solver == "als" and args.variant == "fork":
        ap.error("--solver als solves the squared-error README model; --variant fork (sigmoid cross-entropy, |q_i|) "
                 "is not supported")
    if args.solver == "ials":
        if args.variant == "fork":
            ap.error("--solver ials trains the README model's p_u . q_i; --variant fork (sigmoid cross-entropy, |q_i|) "
                     "is not supported")
        if args.topk <= 0:
            ap.error("--solver ials needs --topk K: the model ranks items, and RMSE against ratings means nothing for it")
        if not (args.alpha >= 0.0 and np.isfinite(args.alpha)):
            ap.error("--alpha must be >= 0 and finite")
    np.random.seed(config.SEED)  # svd_train_val.py:15
    train, val = load(args)
    dict(adam=svd, als=svd_als, ials=svd_ials)[args.solver](train, val, args)
    print("Done!")


if __name__ == "__main__":
    main()
