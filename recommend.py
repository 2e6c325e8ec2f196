"""Top-k recommendations for given users from a checkpoint written by svd_train_val.py.

    python recommend.py --checkpoint fm.ckpt --users 3,17,42 --k 10                  # synthetic ml1m training split
    python recommend.py --checkpoint fm.ckpt --users 3 --dataset mydata --no-exclude
    python recommend.py --checkpoint fm.ckpt --fold-in new_users.csv --k 10            # users not in the checkpoint
    python recommend.py --checkpoint fm.ckpt --similar-items 3,17,42 --k 10           # items like these items

The model (shape and variant) comes from the checkpoint (SvdEngine.from_checkpoint); the path resolves as
svd_train_val.py writes it, under config.BASE_DIR.  Unless --no-exclude is given, the items each user rated in the
training split are never recommended: the split is svd_train_val.load with the same data flags (--dataset, or --synthetic
with --ratings; the synthetic variant follows the checkpoint's model).  The ranking is the exact float64 one of
SvdEngine.rank_users.

--fold-in FILE ranks users the model was not trained on: FILE is a CSV with the header `user,item,rating`, where user is
any label.  Each distinct label is folded into the model from its ratings (SvdEngine.fold_in: the least-squares user row
against the checkpoint's item side, regularised by --reg, the training default of svd_train_val.py --reg) and ranked by
SvdEngine.rank_folded; unless --no-exclude is given, a label's own rated items are never recommended.  No training split is
read.

--similar-items ITEMS lists, for each given item, the items most like it by cosine of the item rows
(SvdEngine.similar_items: exact float64, never the item itself).  No training split is read.

stdout: one line per query user, in the order given (--fold-in: per distinct label, in order of first appearance):
`user<TAB>item:score item:score ...` (scores %.6f; a user with fewer than k rankable items gets fewer pairs, a label that
could not be folded in gets none and a note on stderr); --similar-items: `item<TAB>item:score ...`, one line per given
item.  Everything else goes to stderr.
"""
import argparse
import csv
import os
import sys
from contextlib import redirect_stdout

import numpy as np

import tf_recomm_b200  # noqa: F401
from tf_recomm_b200 import _lib, config, synthetic
from tf_recomm_b200.engine import SvdEngine


def main(argv=None, out=None):
    out = out if out is not None else sys.stdout
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--checkpoint", type=str, default="fm.ckpt", help="as given to svd_train_val.py --checkpoint")
    who = ap.add_mutually_exclusive_group(required=True)
    who.add_argument("--users", type=str, help="comma-separated user ids")
    who.add_argument("--fold-in", dest="fold_in", type=str, default=None,
                     help="CSV with header user,item,rating: rank these users, folded into the model from their ratings")
    who.add_argument("--similar-items", dest="similar_items", type=str, default=None,
                     help="comma-separated item ids: list the items most like each of them (cosine of the item rows)")
    ap.add_argument("--reg", type=float, default=config.LAMBDA_REG,
                    help="L2 weight of the fold-in (the model's training reg; checkpoints do not record it)")
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--dataset", type=str, default=None, help="data/<name>/{train,val,test}.csv (dataio.get_data)")
    ap.add_argument("--synthetic", type=str, default="ml1m", choices=sorted(synthetic.SHAPES))
    ap.add_argument("--ratings", type=int, default=None, help="override the number of synthetic ratings")
    ap.add_argument("--no-exclude", dest="no_exclude", action="store_true",
                    help="rank every item, including the ones the user rated in training")
    args = ap.parse_args(argv)
    if args.fold_in is not None:
        return fold_in(args, out)
    if args.similar_items is not None:
        return similar_items(args, out)
    users = np.array([int(x) for x in args.users.split(",") if x.strip()], np.int64)
    eng = SvdEngine.from_checkpoint(os.path.join(config.BASE_DIR, args.checkpoint))
    exclude = None
    if not args.no_exclude:
        import svd_train_val
        args.variant = "fork" if eng.flags & _lib.LOSS_SIGMOID_CE else "readme"
        args.user_num, args.item_num = eng.U, eng.I
        with redirect_stdout(sys.stderr):   # load() prints the split shapes
            train, _ = svd_train_val.load(args)
        exclude = eng.pair_csr(train["user"], train["item"])
    idx, val = eng.rank_users(users, k=args.k, exclude=exclude)
    idx, val = idx.cpu().numpy(), val.cpu().numpy()
    for u, row_i, row_v in zip(users, idx, val):
        out.write("%d\t%s\n" % (u, " ".join("%d:%.6f" % (i, v) for i, v in zip(row_i, row_v) if i >= 0)))
    out.flush()


def read_ratings(path):
    """CSV `user,item,rating` -> (labels in order of first appearance, row of every rating, items, ratings)."""
    with open(path, newline="") as f:
        rd = csv.reader(f)
        header = [h.strip() for h in next(rd, [])]
        if header != ["user", "item", "rating"]:
            raise SystemExit("%s: expected the header user,item,rating, got %s" % (path, ",".join(header)))
        labels, row_of, rows, items, rates = [], {}, [], [], []
        for rec in rd:
            if not rec:
                continue
            label, item, rating = (x.strip() for x in rec)
            if label not in row_of:
                row_of[label] = len(labels)
                labels.append(label)
            rows.append(row_of[label])
            items.append(int(item))
            rates.append(float(rating))
    return labels, np.array(rows, np.int64), np.array(items, np.int64), np.array(rates, np.float32)


def fold_in(args, out):
    labels, rows, items, rates = read_ratings(args.fold_in)
    eng = SvdEngine.from_checkpoint(os.path.join(config.BASE_DIR, args.checkpoint))
    folded = eng.fold_in(rows, items, rates, n=len(labels), reg=args.reg)
    idx, val = eng.rank_folded(folded, k=args.k, exclude_rated=not args.no_exclude)
    idx, val, info = idx.cpu().numpy(), val.cpu().numpy(), folded.info.cpu().numpy()
    for label, row_i, row_v, st in zip(labels, idx, val, info):
        if st != 0:
            print("user %s: could not be folded in (info %d): no recommendations" % (label, st), file=sys.stderr)
        out.write("%s\t%s\n" % (label, " ".join("%d:%.6f" % (i, v) for i, v in zip(row_i, row_v) if i >= 0)))
    out.flush()


def similar_items(args, out):
    items = np.array([int(x) for x in args.similar_items.split(",") if x.strip()], np.int64)
    eng = SvdEngine.from_checkpoint(os.path.join(config.BASE_DIR, args.checkpoint))
    idx, val = eng.similar_items(items, k=args.k)
    idx, val = idx.cpu().numpy(), val.cpu().numpy()
    for i, row_i, row_v in zip(items, idx, val):
        out.write("%d\t%s\n" % (i, " ".join("%d:%.6f" % (j, v) for j, v in zip(row_i, row_v) if j >= 0)))
    out.flush()


if __name__ == "__main__":
    main()
