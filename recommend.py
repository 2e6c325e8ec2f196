"""Top-k recommendations for given users from a checkpoint written by svd_train_val.py.

    python recommend.py --checkpoint fm.ckpt --users 3,17,42 --k 10                  # synthetic ml1m training split
    python recommend.py --checkpoint fm.ckpt --users 3 --dataset mydata --no-exclude

The model (shape and variant) comes from the checkpoint (SvdEngine.from_checkpoint); the path resolves as
svd_train_val.py writes it, under config.BASE_DIR.  Unless --no-exclude is given, the items each user rated in the
training split are never recommended: the split is svd_train_val.load with the same data flags (--dataset, or --synthetic
with --ratings; the synthetic variant follows the checkpoint's model).  The ranking is the exact float64 one of
SvdEngine.rank_users.

stdout: one line per query user, in the order given: `user<TAB>item:score item:score ...` (scores %.6f; a user with fewer
than k rankable items gets fewer pairs).  Everything else goes to stderr.
"""
import argparse
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
    ap.add_argument("--users", type=str, required=True, help="comma-separated user ids")
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--dataset", type=str, default=None, help="data/<name>/{train,val,test}.csv (dataio.get_data)")
    ap.add_argument("--synthetic", type=str, default="ml1m", choices=sorted(synthetic.SHAPES))
    ap.add_argument("--ratings", type=int, default=None, help="override the number of synthetic ratings")
    ap.add_argument("--no-exclude", dest="no_exclude", action="store_true",
                    help="rank every item, including the ones the user rated in training")
    args = ap.parse_args(argv)
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


if __name__ == "__main__":
    main()
