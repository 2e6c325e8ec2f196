"""SvdEngine: the device-resident state of the matrix-factorization model and the calls that step it.

It owns what the TensorFlow session owned in the reference (the five variables of ops.py:8-12,29-32, the
Adam slots, global_step -- svd_train_val.py:47-56) as CUDA tensors, and drives libtfrecomm.so through
ctypes.  torch is plumbing here (device memory, streams, pinned staging); all arithmetic of the path is in
the hand-written kernels.  No CPU fallback: constructing an engine without CUDA raises.
"""
import contextlib
import ctypes as C
import os
import time
from typing import NamedTuple

import numpy as np
import torch

from . import _lib
from ._lib import (ABS_ITEM, FORK_FLAGS, LOSS_SIGMOID_CE, OPT_SGD, README_FLAGS, REG_BIAS, VAR_ALL, OptScalars, StepWs,
                   SvdTables, TfrError, check)

TABLE_NAMES = ("mu", "user_bias", "item_bias", "user_feat", "item_feat")
_SLOT_FIELDS = {"mu": ("m_mu", "v_mu"), "user_bias": ("m_ub", "v_ub"), "item_bias": ("m_ib", "v_ib"),
                "user_feat": ("m_uf", "v_uf"), "item_feat": ("m_if", "v_if")}


class PairCSR(NamedTuple):
    """(user, item) pairs as CSR by user on the device: indptr int64 [U + 1], items int32 ascending inside a user."""
    indptr: torch.Tensor
    items: torch.Tensor


class FoldedUsers(NamedTuple):
    """Users folded into a trained model (SvdEngine.fold_in), on the device: feat [n, d] / bias [n] fp32, the row's
    least-squares user row; ratings: the fold-in ratings as a PairCSR over the n rows (duplicates kept); info [n] int32,
    0 = ok, j + 1 = pivot j was not > 0, -1 = an item id out of range (rows with info != 0 are NaN)."""
    feat: torch.Tensor
    bias: torch.Tensor
    ratings: PairCSR
    info: torch.Tensor


def _require_cuda():
    if not torch.cuda.is_available():
        raise TfrError("tf-recomm_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback for this path")


class SvdEngine:
    def __init__(self, user_num, item_num, dim, lr, reg, flags=README_FLAGS, var_mask=VAR_ALL, beta1=0.9,
                 beta2=0.999, eps=1e-8, tables=None, device=None, device_init_seed=None):
        """tables: dict of numpy arrays (mu, user_bias, item_bias, user_feat, item_feat) to inject; if None the
        tables are drawn ON THE DEVICE (truncated normal 0.02 / zeros biases) -- for shapes too large to stage
        through host memory (100M x 128)."""
        _require_cuda()
        self.L = _lib.load()
        self.device = torch.device(device if device is not None else "cuda:%d" % torch.cuda.current_device())
        self._dev_index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self.U, self.I, self.d = int(user_num), int(item_num), int(dim)
        self.flags, self.var_mask = int(flags), int(var_mask)
        self.sgd = bool(flags & OPT_SGD)
        self.hyper = dict(lr=float(lr), reg=float(reg), beta1=float(beta1), beta2=float(beta2), eps=float(eps))
        dev = self.device
        with torch.cuda.device(dev):
            self.t, self.slots = {}, {}
            # Feature tables (Adam mode): INTERLEAVED [rows][var | m | v][dim] -- the row of a parameter table and the
            # rows of its two Adam slots are adjacent, so the table-wide pass reads and writes one stream instead of
            # three (tfr_svd_tables.feat_stride = 3*dim).  self.t[...] / self.slots[...] are strided VIEWS of it with
            # the reference's shapes [rows, dim].  SGD mode has no slots: plain [rows][dim].
            self.feat_stride = 0 if self.sgd else 3 * self.d
            for n, rows in (("user_feat", self.U), ("item_feat", self.I)):
                if self.sgd:
                    self.t[n] = torch.empty(rows, self.d, device=dev)
                else:
                    blk = torch.zeros(rows, 3, self.d, device=dev)
                    self.t[n], self.slots["m_" + n], self.slots["v_" + n] = blk[:, 0], blk[:, 1], blk[:, 2]
            if tables is not None:
                for n in TABLE_NAMES:
                    a = np.ascontiguousarray(tables[n], dtype=np.float32)
                    src = torch.from_numpy(a.reshape(-1) if n == "mu" else a)
                    if n in self.t:
                        assert tuple(src.shape) == tuple(self.t[n].shape), (n, src.shape, self.t[n].shape)
                        self.t[n].copy_(src)
                    else:
                        self.t[n] = src.to(dev).contiguous()
            else:
                g = torch.Generator(device=dev)
                g.manual_seed(13575 if device_init_seed is None else int(device_init_seed))
                self.t["mu"] = torch.zeros(1, device=dev)
                self.t["user_bias"] = torch.zeros(self.U, device=dev)
                self.t["item_bias"] = torch.zeros(self.I, device=dev)
                for n in ("user_feat", "item_feat"):
                    # drawn contiguously, then copied into the strided view (trunc_normal_'s in-place math on a view of
                    # a 100M-row table would materialise temporaries anyway); chunked to bound the extra memory
                    rows = self.t[n].shape[0]
                    step = max(1, min(rows, (1 << 28) // max(self.d, 1)))
                    for r0 in range(0, rows, step):
                        tmp = torch.empty(min(step, rows - r0), self.d, device=dev)
                        torch.nn.init.trunc_normal_(tmp, mean=0.0, std=0.02, a=-0.04, b=0.04, generator=g)
                        self.t[n][r0:r0 + tmp.shape[0]].copy_(tmp)
                        del tmp
            assert self.t["user_feat"].shape == (self.U, self.d) and self.t["item_feat"].shape == (self.I, self.d)
            if not self.sgd:
                for n in ("mu", "user_bias", "item_bias"):
                    self.slots["m_" + n] = torch.zeros_like(self.t[n])
                    self.slots["v_" + n] = torch.zeros_like(self.t[n])
            # row -> slot maps: (step stamp << 32 | index of the row's summed gradient); an entry counts only in the
            # step that wrote it, so nothing is reset between steps
            self.user_slot = torch.full((self.U,), -1, dtype=torch.int64, device=dev)
            self.item_slot = torch.full((self.I,), -1, dtype=torch.int64, device=dev)
            self.opt = torch.zeros(C.sizeof(OptScalars), dtype=torch.uint8, device=dev)
            # side stream for the id sort (runs next to the forward): see tfr_svd_train_step
            self.side_streams = [torch.cuda.Stream(device=dev)]
            self._side_arr = (C.c_void_p * 1)(*[s_.cuda_stream for s_ in self.side_streams])
            # fork / join events of the step's side-stream fork: owned by this engine, on this engine's device
            self._fj_events = (C.c_void_p * 2)()
            for k_ in range(2):
                ev = C.c_void_p()
                check(self.L.tfr_event_create(C.byref(ev)))
                self._fj_events[k_] = ev.value
            self._fill_struct()
            check(self.L.tfr_opt_init(self.opt.data_ptr(), lr, reg, beta1, beta2, eps, self.flags, self.var_mask,
                                      self._stream()))
        self._ws = {}
        self._stage = {}
        self._graphs = {}
        self._host_state = {}
        self._copy_stream = torch.cuda.Stream(device=self.device)
        # prefetch_host runs on a worker thread (TFR_FEED_WORKER=0: in line, on the caller's thread)
        self.feed_worker = os.environ.get("TFR_FEED_WORKER", "1") != "0"
        self._feed_pool = None
        self.feed_graphs = os.environ.get("TFR_FEED_GRAPHS", "1") != "0"   # 0: the host-fed step as eager launches
        self._feed_cap = None
        self.host_prof = None       # dict: train_step_host accumulates its host-side phases (seconds) into it
        self.data = None
        self.se_ring = None
        self.overlap = True
        self._primed = None
        self.graph_steps = 8   # steps per captured graph in run_stream_steps (pipelined mode)

    # ---- plumbing ---------------------------------------------------------------------------------------
    def _n_side(self):
        """How many side streams the step may fork onto (self.overlap: True = 1, False = 0)."""
        return 1 if self.overlap else 0

    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def _on_device(self):
        """torch.cuda.device(self.device), or nothing at all when that already is the current device (the context
        manager costs several microseconds per entry: too much for the per-step path of a 30 us step)."""
        if torch.cuda.current_device() == self._dev_index:
            return contextlib.nullcontext()
        return torch.cuda.device(self.device)

    def _fill_struct(self):
        s = SvdTables()
        s.user_num, s.item_num, s.dim = self.U, self.I, self.d
        s.feat_stride = self.feat_stride
        s.mu, s.user_bias, s.item_bias = (self.t[n].data_ptr() for n in ("mu", "user_bias", "item_bias"))
        s.user_feat, s.item_feat = self.t["user_feat"].data_ptr(), self.t["item_feat"].data_ptr()
        if not self.sgd:
            for n, (mf, vf) in _SLOT_FIELDS.items():
                setattr(s, mf, self.slots["m_" + n].data_ptr())
                setattr(s, vf, self.slots["v_" + n].data_ptr())
        s.user_slot, s.item_slot = self.user_slot.data_ptr(), self.item_slot.data_ptr()
        self.tables_struct = s

    def workspace(self, key):
        """Step workspace for batch size `key` (or (B, slot) for the pipelined double buffer)."""
        ws = self._ws.get(key)
        if ws is None:
            B = key[0] if isinstance(key, tuple) else key
            nbytes = check(self.L.tfr_svd_step_workspace_bytes(B, self.d))
            ws = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
            self._ws[key] = ws
        return ws

    def step_ws(self, B):
        ws = self.workspace(B)
        out = StepWs()
        check(self.L.tfr_svd_step_carve(ws.data_ptr(), ws.numel(), B, self.d, C.byref(out)))
        return out

    def _check_ids(self, users, items, n_users=None):
        """ids outside the tables are an error where they enter (TF's CPU embedding_lookup raises
        InvalidArgumentError): nothing out of range ever reaches a gather.  n_users: rows of the user side (default U)."""
        for name, a, n in (("user", users, self.U if n_users is None else n_users), ("item", items, self.I)):
            if isinstance(a, torch.Tensor):
                if a.numel() == 0:
                    continue
                lo, hi = (int(x) for x in torch.aminmax(a))
            else:
                a = np.asarray(a)
                if a.size == 0:
                    continue
                lo, hi = a.min(), a.max()
            if lo < 0 or hi >= n:
                raise TfrError("indices out of range: %s ids span [%s, %s], table has %d rows" % (name, lo, hi, n))

    def _dev_i32(self, a):
        if isinstance(a, torch.Tensor):
            return a.to(device=self.device, dtype=torch.int32).contiguous()
        # the real iterators yield float64 id columns (dataio.py:103); TF's feed casts by value (A.7)
        return torch.from_numpy(np.ascontiguousarray(a).astype(np.int32, copy=False)).to(self.device)

    def _dev_f32(self, a):
        if isinstance(a, torch.Tensor):
            return a.to(device=self.device, dtype=torch.float32).contiguous()
        return torch.from_numpy(np.ascontiguousarray(a).astype(np.float32, copy=False)).to(self.device)

    # ---- forward only: sess.run([logits, infer]) at svd_train_val.py:121-122 --------------------------------
    def forward(self, users, items):
        self._check_ids(users, items)
        users, items = self._dev_i32(users), self._dev_i32(items)
        B = users.numel()
        logits = torch.empty(B, dtype=torch.float32, device=self.device)
        infer = torch.empty(B, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            check(self.L.tfr_svd_forward(C.byref(self.tables_struct), users.data_ptr(), items.data_ptr(), B,
                                         self.flags, logits.data_ptr(), infer.data_ptr(), self._stream()))
        return logits, infer

    # ---- all-pairs scoring: als3.py:110-113 (+ forward.py:47-61 ranking for k = 1) ----------------------------
    def allpairs(self, want_scores=False, want_best=True, use_tensor_cores=None):
        """-> dict(scores [U, I] | None, best_score [U], best_item [U]); tensor cores (tcgen05, tf32) when dim % 32 == 0
        and dim <= 128 unless use_tensor_cores=False (exact fp32 CUDA-core kernel)."""
        if use_tensor_cores is None:
            use_tensor_cores = self.d % 32 == 0 and self.d <= 128
        dev = self.device
        scores = torch.empty(self.U, self.I, dtype=torch.float32, device=dev) if want_scores else None
        bs = torch.empty(self.U, dtype=torch.float32, device=dev) if want_best else None
        bi = torch.empty(self.U, dtype=torch.int32, device=dev) if want_best else None
        nbytes = check(self.L.tfr_allpairs_workspace_bytes(self.U, self.I, self.d, int(use_tensor_cores)))
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        with torch.cuda.device(dev):
            check(self.L.tfr_allpairs(self.t["user_feat"].data_ptr(), self.t["item_feat"].data_ptr(),
                                      self.t["user_bias"].data_ptr(), self.t["item_bias"].data_ptr(),
                                      self.t["mu"].data_ptr(), self.U, self.I, self.d, self.feat_stride,
                                      self.feat_stride, int(use_tensor_cores),
                                      scores.data_ptr() if want_scores else None, bs.data_ptr() if want_best else None,
                                      bi.data_ptr() if want_best else None, ws.data_ptr(), nbytes, self._stream()))
        return dict(scores=scores, best_score=bs, best_item=bi)

    # ---- DISCRETE-branch metrics on the device (svd_train_val.py:94-98,138-143) ----------------------------------------
    def binary_metrics(self, logits, labels):
        """-> dict(nll_sum, n_correct, auc, n_pos, n): summed sigmoid cross-entropy (cost_nll), number of correct
        round(sigmoid(logits)), roc_auc_score(labels, sigmoid(logits)) -- computed on the device (tfr_binary_metrics:
        sort-based AUC reusing the step's radix sort); 32 bytes come back instead of the logits."""
        lg, lb = self._dev_f32(logits), self._dev_f32(labels)
        n = lg.numel()
        nbytes = check(self.L.tfr_binary_metrics_workspace_bytes(n))
        key = ("metrics_ws", nbytes)
        ws = self._stage.get(key)
        if ws is None:
            ws = self._stage[key] = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        out = torch.empty(4, dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            check(self.L.tfr_binary_metrics(lg.data_ptr(), lb.data_ptr(), n, ws.data_ptr(), nbytes, out.data_ptr(),
                                            self._stream()))
        o = out.cpu().numpy()
        return dict(nll_sum=float(o[0]), n_correct=int(round(o[1])), auc=float(o[2]), n_pos=int(round(o[3])), n=n)

    def last_step_metrics(self, B):
        """binary_metrics of the step train_step_host issued LAST, from its device-resident logits and ratings (the
        staging set it used): the DISCRETE branch's per-step train metrics without a second pass over host arrays."""
        hs = self._host_state.get(B)
        if hs is None or hs["last"] is None:
            raise TfrError("no host-fed step of batch size %d has run" % B)
        st = self._host_set(B, hs["last"])   # (never restaged before the next step has been issued: pending <= N_FEED_SETS - 1)
        return self.binary_metrics(st["d_out"][:B], st["d_feed"][2 * B:].view(torch.float32))

    # ---- all-pairs consumers fused into the GEMM epilogue ------------------------------------------------------------
    def _topk_setup(self, k, n_cand):
        k = int(min(k, self.I))
        if n_cand is None:
            n_cand = min(128, max(k + 14, 8))
        dev = self.device
        idx = torch.empty(self.U, k, dtype=torch.int32, device=dev)
        val = torch.empty(self.U, k, dtype=torch.float64, device=dev)
        n_unc = torch.zeros(1, dtype=torch.int32, device=dev)
        nbytes = check(self.L.tfr_allpairs_topk_workspace_bytes(self.U, self.I, k, n_cand))
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        return k, n_cand, idx, val, n_unc, ws, nbytes

    def rank_all_users(self, k=50, n_cand=None, exclude=None):
        """forward.py:47-61 for EVERY user in one sweep of the tcgen05 GEMM: -> (items [U, k] int32, scores [U, k]
        float64, n_uncertified).  Identical to ranking the float64 score matrix of als3.py:112 (score descending, lowest
        item id on ties): tensor-core candidates, float64 rescore, certificate, exact fallback (tfr_allpairs_consume).

        exclude: items each user must not be recommended (usually the training pairs): a (users, items) pair of id arrays
        (host or device) or a PairCSR from pair_csr().  The ranking is then over each user's remaining items
        (tfr_allpairs_rank_excluding); a user with fewer than k of them gets (-inf, -1) past the last one.  With exclude,
        any dim <= 512 is accepted (dims the tensor cores cannot take rank every row exactly on CUDA cores), and an
        engine whose model scores u.|v| (ABS_ITEM, the fork variant) is ranked by that score."""
        if exclude is None:
            k, n_cand, idx, val, n_unc, ws, nbytes = self._topk_setup(k, n_cand)
            with torch.cuda.device(self.device):
                check(self.L.tfr_allpairs_consume(self.t["user_feat"].data_ptr(), self.t["item_feat"].data_ptr(),
                                                  self.t["user_bias"].data_ptr(), self.t["item_bias"].data_ptr(),
                                                  self.t["mu"].data_ptr(), self.U, self.I, self.d, self.feat_stride,
                                                  self.feat_stride, k, n_cand, val.data_ptr(), idx.data_ptr(),
                                                  n_unc.data_ptr(), None, None, None, None, ws.data_ptr(), nbytes,
                                                  self._stream()))
            return idx, val, int(n_unc.item())
        csr = exclude if isinstance(exclude, PairCSR) else self.pair_csr(*exclude)
        return self._rank_excluding(k, n_cand, csr)

    def _rank_excluding(self, k, n_cand, csr):
        """tfr_allpairs_rank_excluding; csr = None: nothing excluded."""
        k, n_cand, idx, val, n_unc, ws, nbytes = self._topk_setup(k, n_cand)
        item_feat, item_stride = self.t["item_feat"], self.feat_stride
        if self.flags & ABS_ITEM:   # the model's score is u.|v| (ops.py:44): rank on a copy of |item_feat|
            item_feat, item_stride = torch.abs(item_feat).contiguous(), 0
        with torch.cuda.device(self.device):
            check(self.L.tfr_allpairs_rank_excluding(
                self.t["user_feat"].data_ptr(), item_feat.data_ptr(), self.t["user_bias"].data_ptr(),
                self.t["item_bias"].data_ptr(), self.t["mu"].data_ptr(), self.U, self.I, self.d, self.feat_stride,
                item_stride, k, n_cand, csr.indptr.data_ptr() if csr is not None else None,
                csr.items.data_ptr() if csr is not None else None, val.data_ptr(), idx.data_ptr(), n_unc.data_ptr(),
                ws.data_ptr(), nbytes, self._stream()))
        return idx, val, int(n_unc.item())

    def rank_users(self, users, k=50, exclude=None):
        """forward.py:47-61 for the users asked about: -> (items [n, k] int32, scores [n, k] float64) on the device, row q
        the ranking of users[q] (ids may repeat, any order; host or device), k = min(k, I).  Bit for bit the user's row of
        rank_all_users(k, exclude=exclude), at a cost that scales with n instead of U (tfr_rank_users: float64 on CUDA
        cores).  exclude: (users, items) pairs or a PairCSR from pair_csr(), indexed by user id; build it once for repeated
        calls.  The fork model (ABS_ITEM) is ranked by u.|v| + biases."""
        self._check_ids(users, [])
        csr = None
        if exclude is not None:
            csr = exclude if isinstance(exclude, PairCSR) else self.pair_csr(*exclude)
        q = self._dev_i32(np.atleast_1d(np.asarray(users)) if not isinstance(users, torch.Tensor) else users.reshape(-1))
        return self._rank_rows(self.t["user_feat"], self.t["user_bias"], self.U, self.feat_stride, q, k, csr)

    def _rank_rows(self, user_feat, user_bias, n_users, user_stride, q, k, csr):
        """tfr_rank_users of the query rows q (device int32) of the user table (user_feat, user_bias) against this
        engine's item side; csr: exclusion CSR indexed by the table's rows, or None."""
        n, k = int(q.numel()), int(min(k, self.I))
        dev = self.device
        idx = torch.empty(n, k, dtype=torch.int32, device=dev)
        val = torch.empty(n, k, dtype=torch.float64, device=dev)
        if n == 0:
            return idx, val
        nbytes = check(self.L.tfr_rank_users_workspace_bytes(n, self.I, k))
        key = ("rank_users_ws", n, k)   # serving calls of one shape reuse their workspace
        ws = self._stage.get(key)
        if ws is None:
            ws = self._stage[key] = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        with torch.cuda.device(dev):
            check(self.L.tfr_rank_users(
                user_feat.data_ptr(), self.t["item_feat"].data_ptr(), user_bias.data_ptr(),
                self.t["item_bias"].data_ptr(), self.t["mu"].data_ptr(), n_users, self.I, self.d, user_stride,
                self.feat_stride, self.flags & ABS_ITEM, q.data_ptr(), n, k,
                csr.indptr.data_ptr() if csr is not None else None, csr.items.data_ptr() if csr is not None else None,
                val.data_ptr(), idx.data_ptr(), ws.data_ptr(), nbytes, self._stream()))
        return idx, val

    # ---- fold-in: user rows for users the model was not trained on ------------------------------------------------------
    def fold_in(self, rows, items, rates, n=None, reg=None):
        """Least-squares user rows for new users (or new ratings of known ones) against the trained item side: for each
        row label r in [0, n) the (p_u, b_u) that minimises the training loss (ops.py:81-89,124-126, squared error +
        reg * L2) over the ratings (rows == r) with item_feat, item_bias and mu fixed -- tfr_fold_in_users, float64 normal
        equations solved by Cholesky on the device.  rows / items / rates: host or device arrays of one rating each
        (duplicates count, as in training); n defaults to max(rows) + 1; reg defaults to the engine's reg.  A row without
        ratings gets p = 0, b = 0.  -> FoldedUsers (rank it with rank_folded).  The fork's sigmoid-CE loss is not a
        least-squares problem and is refused."""
        if self.flags & LOSS_SIGMOID_CE:
            raise TfrError("fold_in solves the squared-error objective; the sigmoid cross-entropy model is not supported")
        reg = self.hyper["reg"] if reg is None else float(reg)
        if not reg >= 0.0:
            raise TfrError("fold_in: reg must be >= 0, got %r" % reg)
        sizes = [a.numel() if isinstance(a, torch.Tensor) else np.asarray(a).size for a in (rows, items, rates)]
        if len(set(sizes)) != 1:
            raise TfrError("fold_in: rows, items and rates differ in length: %s" % sizes)
        if n is None:
            n = int((rows if isinstance(rows, torch.Tensor) else np.asarray(rows)).max()) + 1 if sizes[0] else 0
        n = int(n)
        indptr, it, rt = self._csr_by_user(rows, items, rates, n_rows=n)
        dev = self.device
        feat = torch.empty(n, self.d, dtype=torch.float32, device=dev)
        bias = torch.empty(n, dtype=torch.float32, device=dev)
        info = torch.empty(n, dtype=torch.int32, device=dev)
        with torch.cuda.device(dev):
            check(self.L.tfr_fold_in_users(
                self.t["item_feat"].data_ptr(), self.t["item_bias"].data_ptr(), self.t["mu"].data_ptr(), self.I, self.d,
                self.feat_stride, self.flags, reg, indptr.data_ptr(), it.data_ptr(), rt.data_ptr(), n, feat.data_ptr(),
                bias.data_ptr(), info.data_ptr(), self._stream()))
        return FoldedUsers(feat, bias, PairCSR(indptr, it), info)

    def rank_folded(self, folded, k=50, exclude_rated=True):
        """Top-k of folded users (fold_in): -> (items [n, k] int32, scores [n, k] float64) on the device, row r the ranking
        of folded row r, scored as rank_users scores a trained user (tfr_rank_users on the folded rows as an n-row user
        table; u.|v| for the fork model).  exclude_rated: never recommend the items the row was folded in from.  A row
        that could not be folded (info != 0, NaN) ranks nothing: (-inf, -1)."""
        n = int(folded.feat.shape[0])
        q = torch.arange(n, dtype=torch.int32, device=self.device)
        return self._rank_rows(folded.feat, folded.bias, n, 0, q, k, folded.ratings if exclude_rated else None)

    def _csr_by_user(self, users, items, rates=None, dedup=False, n_rows=None):
        """(user, item[, rate]) pairs -> CSR by user, item ids ascending inside a user: (indptr int64 [U + 1], items int32,
        rates float32 | None).  dedup: every distinct pair once (rates are then not carried); otherwise every pair as
        given, duplicates included, in a stable order.  n_rows: rows of the CSR (user ids in [0, n_rows)), default U."""
        self._check_ids(users, items, n_rows)
        n_rows = self.U if n_rows is None else n_rows
        dev = self.device
        u, i = self._dev_i32(users).to(torch.int64), self._dev_i32(items).to(torch.int64)
        rt = None
        if dedup:
            key = torch.unique(u * self.I + i)   # sorted
            u, it = key // self.I, (key % self.I).to(torch.int32).contiguous()
        else:
            r = self._dev_f32(rates) if rates is not None else None
            order = torch.argsort(u * self.I + i, stable=True)
            it = i[order].to(torch.int32).contiguous()
            rt = r[order].contiguous() if r is not None else None
        indptr = torch.zeros(n_rows + 1, dtype=torch.int64, device=dev)
        indptr[1:] = torch.cumsum(torch.bincount(u, minlength=n_rows), 0)
        return indptr, it, rt

    def pair_csr(self, users, items):
        """The distinct (user, item) pairs as a PairCSR: build an exclusion set once, pass it to rank_all_users /
        ranking_metrics as often as needed."""
        indptr, it, _ = self._csr_by_user(users, items, dedup=True)
        return PairCSR(indptr, it)

    def ranking_metrics(self, k, users, items, rates=None, min_rating=None, exclude=None, n_cand=None):
        """Top-k recommendation quality on held-out pairs: every user is ranked over the items not in `exclude` (usually
        the training pairs; (users, items) or a PairCSR), and the ranking is scored against the user's relevant items =
        the distinct held-out pairs (users, items) -- with rates >= min_rating when both are given -- minus any pair in
        `exclude` (an excluded item can never be recommended).  Users without relevant items are not evaluated.
        -> dict(hr, precision, recall, ndcg, n_users, n_uncertified): means over the evaluated users (hit rate, precision,
        recall and NDCG at k, tfr_ranking_metrics on the device), n_users = how many were evaluated."""
        excl = None
        if exclude is not None:
            excl = exclude if isinstance(exclude, PairCSR) else self.pair_csr(*exclude)
        self._check_ids(users, items)
        if rates is not None and min_rating is not None:
            keep = self._dev_f32(rates) >= float(min_rating)
            users, items = self._dev_i32(users)[keep], self._dev_i32(items)[keep]
        dev = self.device
        key = torch.unique(self._dev_i32(users).to(torch.int64) * self.I + self._dev_i32(items).to(torch.int64))
        if excl is not None and excl.items.numel() > 0:
            ex_user = torch.repeat_interleave(torch.arange(self.U, device=dev), excl.indptr[1:] - excl.indptr[:-1])
            ex_key = ex_user * self.I + excl.items.to(torch.int64)   # sorted: CSR order
            pos = torch.searchsorted(ex_key, key).clamp_(max=ex_key.numel() - 1)
            key = key[ex_key[pos] != key]
        rel_indptr = torch.zeros(self.U + 1, dtype=torch.int64, device=dev)
        rel_indptr[1:] = torch.cumsum(torch.bincount(key // self.I, minlength=self.U), 0)
        rel_item = (key % self.I).to(torch.int32).contiguous()
        idx, _, n_unc = self._rank_excluding(k, n_cand, excl)
        s = self.ranking_sums(idx, PairCSR(rel_indptr, rel_item)).cpu().numpy()
        n = int(round(s[4]))
        mean = (lambda x: float(x) / n) if n else (lambda x: float("nan"))
        return dict(hr=mean(s[0]), precision=mean(s[1]), recall=mean(s[2]), ndcg=mean(s[3]), n_users=n,
                    n_uncertified=n_unc)

    def ranking_sums(self, topk_idx, relevant, row_metrics=None):
        """tfr_ranking_metrics of a ranking topk_idx [n, k] (int32, device) against relevant, a PairCSR over the same n
        rows -> (sum HR, sum precision, sum recall, sum NDCG, rows evaluated), float64 [5] on the device; row_metrics: a
        float64 [n, 4] device tensor to receive the per-row values (NaN where not evaluated)."""
        n, k = topk_idx.shape
        dev = self.device
        sums = torch.empty(5, dtype=torch.float64, device=dev)
        nbytes = check(self.L.tfr_ranking_metrics_workspace_bytes(n, k))
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        with torch.cuda.device(dev):
            check(self.L.tfr_ranking_metrics(topk_idx.data_ptr(), n, k, relevant.indptr.data_ptr(),
                                             relevant.items.data_ptr(),
                                             row_metrics.data_ptr() if row_metrics is not None else None, sums.data_ptr(),
                                             ws.data_ptr(), nbytes, self._stream()))
        return sums

    def observed_rmse(self, users, items, rates):
        """als3.py:110-120,139-143: RMSE of M[user_ids, work_ids] against the ratings, with M = U.V^T + biases consumed
        tile by tile in the GEMM epilogue (never materialised).  -> (rmse, row_se [U] float64)."""
        dev = self.device
        indptr, it, rt = self._csr_by_user(users, items, rates)
        row_se = torch.empty(self.U, dtype=torch.float64, device=dev)
        with torch.cuda.device(dev):
            check(self.L.tfr_allpairs_consume(self.t["user_feat"].data_ptr(), self.t["item_feat"].data_ptr(),
                                              self.t["user_bias"].data_ptr(), self.t["item_bias"].data_ptr(),
                                              self.t["mu"].data_ptr(), self.U, self.I, self.d, self.feat_stride,
                                              self.feat_stride, 0, 0, None, None, None, indptr.data_ptr(), it.data_ptr(),
                                              rt.data_ptr(), row_se.data_ptr(), None, 0, self._stream()))
        n = max(int(it.numel()), 1)
        return float(torch.sqrt(row_se.sum() / n)), row_se

    # ---- ranking: forward.py:47-61 get_ranking (every item scored for one user, sorted, first 50 kept) --------------
    def get_ranking(self, users, k=50):
        """-> (items [n, k] int32, scores [n, k]) for a user id or a sequence of them: the k best items of each user in
        rank order (ties: lowest item id), scored exactly (fp32 forward over all items, tfr_svd_forward's logits)."""
        users = np.atleast_1d(np.asarray(users)).astype(np.int64)
        n, k = len(users), int(min(k, self.I))
        dev = self.device
        uu = torch.from_numpy(np.repeat(users, self.I).astype(np.int32)).to(dev)
        ii = torch.arange(self.I, dtype=torch.int32, device=dev).repeat(n)
        scores = torch.empty(n * self.I, dtype=torch.float32, device=dev)
        vals = torch.empty(n, k, dtype=torch.float32, device=dev)
        idx = torch.empty(n, k, dtype=torch.int32, device=dev)
        with torch.cuda.device(dev):
            check(self.L.tfr_svd_forward(C.byref(self.tables_struct), uu.data_ptr(), ii.data_ptr(), n * self.I, self.flags,
                                         scores.data_ptr(), None, self._stream()))
            check(self.L.tfr_topk_rows(scores.data_ptr(), n, self.I, self.I, k, vals.data_ptr(), idx.data_ptr(),
                                       self._stream()))
        return idx, vals

    # ---- one train step on a device-resident batch: sess.run([train_op, logits, infer]), :70-72 -------------
    def train_step(self, users, items, rates, logits=None, infer=None, check_ids=True):
        if check_ids:
            self._check_ids(users, items)
        users, items, rates = self._dev_i32(users), self._dev_i32(items), self._dev_f32(rates)
        B = users.numel()
        if logits is None:
            logits = torch.empty(B, dtype=torch.float32, device=self.device)
        if infer is None:
            infer = torch.empty(B, dtype=torch.float32, device=self.device)
        ws = self.workspace(B)
        with torch.cuda.device(self.device):
            st = self._stream()  # (lr_t of this step was left behind by the previous step's finish / tfr_opt_init)
            check(self.L.tfr_svd_train_step(C.byref(self.tables_struct), self.opt.data_ptr(), users.data_ptr(),
                                            items.data_ptr(), rates.data_ptr(), B, logits.data_ptr(),
                                            infer.data_ptr(), self.flags, self.var_mask, ws.data_ptr(), ws.numel(),
                                            st, self._side_arr, self._n_side(), self._fj_events))
        return logits, infer

    # ---- host-fed step (the feed_dict path): pinned staging, H2D, step, D2H of the fetched predictions -------
    _FEED_DTYPES = {np.dtype(np.float64): 0, np.dtype(np.float32): 1, np.dtype(np.int32): 2, np.dtype(np.int64): 3}

    def _feed_col(self, a):
        """(host pointer, dtype code, byte stride) of a 1-D column for tfr_host_pack_feed; anything exotic is first
        converted to float64 (what the reference's iterators yield, dataio.py:103)."""
        a = np.asarray(a)
        if a.ndim != 1 or a.dtype not in self._FEED_DTYPES:
            a = np.ascontiguousarray(a, dtype=np.float64).reshape(-1)
        return a, a.ctypes.data, self._FEED_DTYPES[a.dtype], (a.strides[0] if a.size else a.itemsize)

    # The feed path is a ring of staging sets (include/tfrecomm.h, "the feed_dict step").  prefetch_host(batch) hands a
    # coming batch to the feed worker thread, which packs its columns into the set's pinned buffer (value cast + range check
    # in C; no stream is touched).  train_step_host(batch) launches the set's step GRAPH: forward + segment sums, then the
    # table pass, and beside the pass one branch of kernels that delivers the predictions (they come from the PRE-update
    # tables, SURVEY A.7) into pinned memory, fetches the staged NEXT batch from its pinned buffer and sorts its ids; it
    # returns as soon as the delivery flag says the predictions are on the host.  A driver that owns its iterator
    # (svd_train_val.py) hands over batches t+1 .. t+3 BEFORE it asks for step t (up to four may be pending: one stepping,
    # one being fetched + sorted, two packed or being packed -- the slack that keeps a late pack from ever reaching the step
    # stream; profiles/r02_feed_path.md has the measurements behind every one of these choices).  A plain
    # sess.run(feed_dict) without a prefetch does the same work in line: pack, eager copy + sort, the step graph without
    # a next batch.  Every reuse of a staging set is ordered: the pinned buffer is never repacked before the step that
    # consumed it has finished, the device buffers never overwritten while a step still reads them (stream order inside
    # the graphs, the set's events on the eager path -- fetch=False and TFR_FEED_GRAPHS=0 use only that one).
    N_FEED_SETS = 5

    def _host_set(self, B, k):
        key = ("host", B, k)
        st = self._stage.get(key)
        if st is None:
            ws = self.workspace((B, "h", k))
            fs = _lib.FeedSet()
            st = dict(h_feed=torch.empty(3 * B, dtype=torch.int32).pin_memory(),
                      d_feed=torch.empty(3 * B, dtype=torch.int32, device=self.device),
                      d_out=torch.empty(2 * B, dtype=torch.float32, device=self.device),
                      h_out=torch.empty(2 * B, dtype=torch.float32).pin_memory(), ws=ws, fs=fs, events=[],
                      d_sync=torch.zeros(2, dtype=torch.int32, device=self.device),
                      h_flag=torch.zeros(16, dtype=torch.int32).pin_memory())
            fs.h_feed, fs.d_feed = st["h_feed"].data_ptr(), st["d_feed"].data_ptr()
            fs.d_out, fs.h_out = st["d_out"].data_ptr(), st["h_out"].data_ptr()
            fs.workspace, fs.workspace_bytes = ws.data_ptr(), ws.numel()
            fs.d_sync, fs.h_flag = st["d_sync"].data_ptr(), st["h_flag"].data_ptr()
            with torch.cuda.device(self.device):
                for f in ("ev_h2d", "ev_sorted", "ev_pred", "ev_d2h", "ev_done"):
                    ev = C.c_void_p()
                    check(self.L.tfr_event_create(C.byref(ev)))
                    setattr(fs, f, ev.value)
                    st["events"].append(ev.value)
            self._stage[key] = st
        return st

    def _stage_task(self, st, cols, B):
        """tfr_svd_feed_stage (the host-side pack into the pinned buffer; no stream is touched) on the feed worker thread:
        ctypes releases the GIL for the call, so the packing of a coming batch (the one piece of real host work of a
        step) overlaps the main thread's launch / wait / copy-out.  check() runs here, on the thread that made the call:
        the library's error text is thread-local."""
        (ku, pu, du, su), (ki, pi, di, si), (kr, pr, dr, sr) = cols
        with torch.cuda.device(self.device):
            check(self.L.tfr_svd_feed_stage(C.byref(self.tables_struct), C.byref(st["fs"]), pu, du, su, pi, di, si, pr, dr,
                                            sr, B))

    def prefetch_host(self, users, items, rates, _inline=False):
        """Hands over a coming batch early: it is packed right away (on ONE worker thread, in order); its H2D copy and id
        sort are issued by the step before it, beside that step's forward and table pass.  Up to N_FEED_SETS - 1 batches
        may be pending; they must be stepped in the order they were handed over (train_step_host with these very
        arrays) -- a different batch drops everything that is pending.  Errors of a handed-over batch (ids out of range)
        surface when that batch is stepped."""
        B = len(users)
        hs = self._host_state.setdefault(B, dict(next=0, pending=[], last=None))
        if len(hs["pending"]) >= self.N_FEED_SETS - 1:
            raise TfrError("too many batches pending: step one before prefetching another")
        k = hs["next"]
        hs["next"] = (k + 1) % self.N_FEED_SETS
        st = self._host_set(B, k)
        cols = (self._feed_col(users), self._feed_col(items), self._feed_col(rates))   # (array kept alive, ptr, dtype, stride)
        fut = None
        if self.feed_worker and not _inline:
            if self._feed_pool is None:
                from concurrent.futures import ThreadPoolExecutor
                self._feed_pool = ThreadPoolExecutor(max_workers=1, thread_name_prefix="tfr-feed")
            fut = self._feed_pool.submit(self._stage_task, st, cols, B)
        else:
            self._stage_task(st, cols, B)
        hs["pending"].append(dict(k=k, arrays=(users, items, rates), fut=fut, cols=cols, sorted=False))

    def _sort_pending(self, B, e, after_event):
        """Queues the H2D copy + id sort of a staged batch on the side stream (once it IS staged: the worker's errors are
        raised here)."""
        if e["sorted"]:
            return
        if e["fut"] is not None:
            e["fut"].result()
        e["sorted"] = True
        with torch.cuda.device(self.device):
            check(self.L.tfr_svd_feed_sort(C.byref(self.tables_struct), self.opt.data_ptr(), C.byref(self._host_set(B, e["k"])["fs"]),
                                           B, self.side_streams[0].cuda_stream, after_event))

    def _small_tables(self):
        """The table pass is a few microseconds (the id sort is then the longest thing in a step)."""
        if getattr(self, "prefetch_at_start", None) is not None:
            return bool(self.prefetch_at_start)
        return 24 * (self.U + self.I) * (self.d + 1) < 64e6

    def _feed_graph(self, B, k, k_next, mode):
        """The executable graph of one host-fed step on staging set k (+ copy and sort of the batch staged in k_next)."""
        key = ("feed", B, k, k_next, mode, self.flags, self.var_mask, self._small_tables())
        g = self._graphs.get(key)
        if g is None:
            if self._feed_cap is None:
                self._feed_cap = [torch.cuda.Stream(device=self.device) for _ in range(2)]
            exe = C.c_void_p()
            with torch.cuda.device(self.device):
                check(self.L.tfr_svd_feed_graph_create(
                    C.byref(self.tables_struct), self.opt.data_ptr(), C.byref(self._host_set(B, k)["fs"]),
                    C.byref(self._host_set(B, k_next)["fs"]) if k_next is not None else None, B, self.flags, self.var_mask,
                    mode, int(self._small_tables()), *(x.cuda_stream for x in self._feed_cap), C.byref(exe)))
            g = self._graphs[key] = exe.value
        return g

    def prepare_feed_graphs(self, B, fetch=True):
        """Captures (without running anything) every step graph a host-fed loop of batch size B is going to launch, so that
        no capture / instantiation falls into a timed region: per staging set the graph with the next set's fetch + sort
        and the one without."""
        mode = 0 if not fetch else (1 if not (self.flags & LOSS_SIGMOID_CE) else 2)
        if not self.feed_graphs:
            return
        for k in range(self.N_FEED_SETS):
            self._feed_graph(B, k, None, mode)
            if fetch:
                self._feed_graph(B, k, (k + 1) % self.N_FEED_SETS, mode)

    def train_step_host(self, users, items, rates, fetch=True):
        B = len(users)
        hs = self._host_state.setdefault(B, dict(next=0, pending=[], last=None))
        pend = hs["pending"]
        if not pend or any(x is not y for x, y in zip(pend[0]["arrays"], (users, items, rates))):
            fetched = any(e["sorted"] for e in pend)
            for e in pend:   # not the batch that was handed over: drop what is pending (after its task has run)
                if e["fut"] is not None:
                    e["fut"].exception()
            pend.clear()
            if fetched:   # a step in flight is copying / sorting a dropped batch: let it finish before its set is reused
                torch.cuda.current_stream(self.device).synchronize()
                self.side_streams[0].synchronize()
            self.prefetch_host(users, items, rates, _inline=True)   # nothing to overlap with: no hand-off to the worker
        head = pend.pop(0)
        prof = self.host_prof
        t0 = time.perf_counter() if prof is not None else 0.0
        self._sort_pending(B, head, None)   # (queued by the previous step already when the batch was handed over early)
        st = self._host_set(B, head["k"])
        hs["last"] = head["k"]
        # the README head is the identity (infer == logits): one array goes back instead of two
        identity_head = not (self.flags & LOSS_SIGMOID_CE)
        mode = 0 if not fetch else (1 if identity_head else 2)
        # The next batch's copy + id sort belong beside this step's table pass: not beside its forward + segment sums
        # (which the sort slows), not after the pass (where they are on the critical path).  The step goes down as ONE
        # graph that has them as a branch (tfr_svd_feed_graph_create says why eager side-stream launches do not do);
        # a batch whose packing is still under way is copied + sorted eagerly once the predictions have arrived.
        nxt = pend[0] if pend and not pend[0]["sorted"] else None
        if nxt is not None and nxt["fut"] is not None and not (nxt["fut"].done() and nxt["fut"].exception() is None):
            nxt = None   # still being packed, or failed: its own step deals with it (and raises its error)
        if self.feed_graphs and not fetch:
            # the worker repacks a pinned buffer on the strength of the predictions the host has SEEN (the delivery flag):
            # a step that fetches nothing leaves the next batch's copy + sort to the eager, event-ordered path
            nxt = None
        if nxt is not None:
            nxt["sorted"] = True
        fs_next = C.byref(self._host_set(B, nxt["k"])["fs"]) if nxt is not None else None
        with self._on_device():
            if self.feed_graphs:
                g = self._feed_graph(B, head["k"], nxt["k"] if nxt is not None else None, mode)
                check(self.L.tfr_svd_feed_graph_launch(g, C.byref(st["fs"]), fs_next, mode, self._stream()))
            else:
                check(self.L.tfr_svd_feed_step(C.byref(self.tables_struct), self.opt.data_ptr(), C.byref(st["fs"]), B,
                                               self.flags, self.var_mask, mode, self._stream(),
                                               self._copy_stream.cuda_stream, fs_next, self.side_streams[0].cuda_stream))
        t1 = time.perf_counter() if prof is not None else 0.0
        if not fetch:
            return None
        if self.feed_graphs:   # the delivery kernel's flag in pinned memory
            check(self.L.tfr_host_wait_flag(st["fs"].h_flag, st["fs"].deliver_seq, 30_000_000))
        else:
            check(self.L.tfr_event_synchronize(st["fs"].ev_d2h))
        t2 = time.perf_counter() if prof is not None else 0.0
        if pend and not pend[0]["sorted"] and not (pend[0]["fut"] is not None and pend[0]["fut"].done()
                                                     and pend[0]["fut"].exception() is not None):
            self._sort_pending(B, pend[0], None)
        t3 = time.perf_counter() if prof is not None else 0.0
        if identity_head:
            out = st["h_out"][B:].numpy().copy()   # one copy out of the pinned buffer
            res = (out, out)
        else:
            out = st["h_out"].numpy().copy()
            res = (out[:B], out[B:])
        if prof is not None:   # host-side breakdown for tools/e2e_breakdown.py
            t4 = time.perf_counter()
            for name, dt in (("issue_step", t1 - t0), ("wait_predictions", t2 - t1), ("issue_next_sort", t3 - t2),
                             ("copy_out", t4 - t3)):
                prof[name] = prof.get(name, 0.0) + dt
        return res

    def d2h_bytes(self, B):
        return (4 if not (self.flags & LOSS_SIGMOID_CE) else 8) * B

    h2d_bytes = staticmethod(lambda B: 12 * B)

    # ---- device-resident training data + pre-drawn index stream (dataio.ShuffleIterator on the device) ------
    def set_train_data(self, col_user, col_item, col_rate):
        self._check_ids(col_user, col_item)   # once, where the columns enter: the assembled batches are then in range
        # captured stream graphs bake the column addresses in: drop them (and whatever was assembled ahead)
        self._destroy_graphs()
        self._primed = None
        self.data = dict(user=self._dev_i32(col_user), item=self._dev_i32(col_item), rate=self._dev_f32(col_rate))

    def _destroy_graphs(self):
        for g in self._graphs.values():
            self.L.tfr_graph_destroy(g)
        self._graphs.clear()

    def close(self):
        """Releases the captured graphs (device memory goes with the tensors)."""
        if getattr(self, "_feed_pool", None) is not None:
            self._feed_pool.shutdown(wait=True)
            self._feed_pool = None
        if getattr(self, "_graphs", None):
            torch.cuda.synchronize(self.device)
            self._destroy_graphs()
        for k_ in range(2):
            if getattr(self, "_fj_events", None) is not None and self._fj_events[k_]:
                self.L.tfr_event_destroy(self._fj_events[k_])
                self._fj_events[k_] = None
        for st in getattr(self, "_stage", {}).values():
            if isinstance(st, dict) and st.get("events"):
                for ev in st["events"]:
                    self.L.tfr_event_destroy(ev)
                st["events"] = []

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_index_stream(self, row_index, B):
        """row_index: the reference's np.random.randint(0, N, B) draws for consecutive steps, concatenated."""
        if isinstance(row_index, torch.Tensor):
            ri = row_index.to(device=self.device, dtype=torch.int64).contiguous()
        else:
            ri = torch.from_numpy(np.ascontiguousarray(row_index, dtype=np.int64)).to(self.device)
        assert ri.numel() % B == 0
        # captured graphs bake the buffer's address: keep ONE persistent buffer and copy new streams into it
        # (+ B zero entries of slack: the pipelined step assembles one batch past the end)
        cap = getattr(self, "_row_index_buf", None)
        if cap is None or cap.numel() < ri.numel() + B:
            self._row_index_buf = torch.zeros(ri.numel() + B, dtype=torch.int64, device=self.device)
            self._destroy_graphs()
        self._row_index_buf[:ri.numel()].copy_(ri)
        self._row_index_buf[ri.numel():].zero_()
        self._primed = None
        self.row_index = self._row_index_buf
        self.stream_B = B
        self.set_batch_cursor(0)

    def set_batch_cursor(self, k):
        self._primed = None
        with torch.cuda.device(self.device):
            check(self.L.tfr_opt_set_cursor(self.opt.data_ptr(), int(k), self._stream()))

    def set_se_ring(self, n):
        self.se_ring = torch.zeros(n, dtype=torch.float64, device=self.device)
        check(self.L.tfr_opt_set_se_ring(self.opt.data_ptr(), self.se_ring.data_ptr(), n, self._stream()))

    # ---- debug timeline (in-kernel %globaltimer stamps; there is no nsys on the box) ----------------------
    TL_NAMES = ("assemble", "fwd_err", "sort", "seg_tiles", "seg_fixup", "adam_pass", "-", "-", "-", "sgd_slice",
                "-", "finish")

    def enable_timeline(self):
        self.timeline = torch.zeros(32, dtype=torch.int64, device=self.device)
        check(self.L.tfr_opt_set_timeline(self.opt.data_ptr(), self.timeline.data_ptr(), self._stream()))

    def reset_timeline(self):
        self.timeline[:16] = torch.iinfo(torch.int64).max
        self.timeline[16:] = 0

    def read_timeline(self):
        """{kernel: (start_us, end_us)} relative to the earliest kernel start of the step."""
        t = self.timeline.cpu().numpy()
        begin, end = t[:16], t[16:]
        live = [k for k in range(len(self.TL_NAMES)) if end[k] > 0]
        t0 = min(begin[k] for k in live)
        return {self.TL_NAMES[k]: ((begin[k] - t0) / 1e3, (end[k] - t0) / 1e3) for k in live}

    def _enqueue_stream_step(self, B, bufs, batch_index=-1):
        """assemble -> full step, one batch, everything on the current stream (+ the sort's side stream)."""
        st = self._stream()
        check(self.L.tfr_svd_batch_assemble(C.byref(self.tables_struct), self.opt.data_ptr(),
                                            self.data["user"].data_ptr(), self.data["item"].data_ptr(),
                                            self.data["rate"].data_ptr(), self.row_index.data_ptr(), batch_index, B,
                                            bufs["users"].data_ptr(), bufs["items"].data_ptr(),
                                            bufs["rates"].data_ptr(), st))
        ws = self.workspace(B)
        check(self.L.tfr_svd_train_step(C.byref(self.tables_struct), self.opt.data_ptr(), bufs["users"].data_ptr(),
                                        bufs["items"].data_ptr(), bufs["rates"].data_ptr(), B,
                                        bufs["logits"].data_ptr(), bufs["infer"].data_ptr(), self.flags,
                                        self.var_mask, ws.data_ptr(), ws.numel(), st, self._side_arr, self._n_side(),
                                        self._fj_events))

    def _prefetch(self, B, slot, prime, stream_handle):
        """Assemble + id sort of a batch into buffer set `slot` (tfr_svd_prefetch_batch).  prime: the batch at
        batch_cursor, on the step's own stream, and prefetch_cursor := batch_cursor + 1; otherwise the batch at
        prefetch_cursor (a counter only the side stream advances: the concurrent step's last CTA advances
        batch_cursor, which must therefore not be read here)."""
        bufs, ws = self.stream_buffers(B, slot), self.workspace((B, slot))
        check(self.L.tfr_svd_prefetch_batch(C.byref(self.tables_struct), self.opt.data_ptr(),
                                            self.data["user"].data_ptr(), self.data["item"].data_ptr(),
                                            self.data["rate"].data_ptr(), self.row_index.data_ptr(),
                                            -3 if prime else -2, B,
                                            bufs["users"].data_ptr(), bufs["items"].data_ptr(),
                                            bufs["rates"].data_ptr(), ws.data_ptr(), ws.numel(), stream_handle))

    def _enqueue_pipelined_step(self, B, slot):
        """Step on the batch already assembled + sorted in set `slot`, while the NEXT batch is assembled + sorted
        into the other set on the side stream: the id-only work leaves the critical path (it runs under the
        bandwidth-bound table pass, which it barely disturbs)."""
        main = torch.cuda.current_stream(self.device)
        side = self.side_streams[0]
        bufs, ws = self.stream_buffers(B, slot), self.workspace((B, slot))

        def phase(p):
            check(self.L.tfr_svd_train_step_presorted(C.byref(self.tables_struct), self.opt.data_ptr(),
                                                      bufs["users"].data_ptr(), bufs["items"].data_ptr(),
                                                      bufs["rates"].data_ptr(), B, bufs["logits"].data_ptr(),
                                                      bufs["infer"].data_ptr(), self.flags, self.var_mask, p,
                                                      ws.data_ptr(), ws.numel(), main.cuda_stream))
        # Where to fork the next batch's assemble + sort: UNDER the table pass when that pass is long (it is
        # bandwidth-bound and barely notices them, while the latency-bound gathers of phase 1 would slow down
        # beside them); at the start of the step when the tables are small and the pass is a few microseconds.
        small = self._small_tables()
        if small:
            side.wait_stream(main)
            self._prefetch(B, 1 - slot, False, side.cuda_stream)
        phase(1)                      # forward + segment sums
        if not small:
            side.wait_stream(main)
            self._prefetch(B, 1 - slot, False, side.cuda_stream)
        hook = getattr(self, "timing_hook", None)   # bench.py: event-record nodes around the table pass, in situ
        if hook:
            hook("pass_begin", slot, main)
        phase(2)                      # Adam pass + finish
        if hook:
            hook("pass_end", slot, main)
        main.wait_stream(side)

    def stream_buffers(self, B, slot=0):
        key = ("bufs", B, slot)
        b = self._stage.get(key)
        if b is None:
            dev = self.device
            b = dict(users=torch.empty(B, dtype=torch.int32, device=dev),
                     items=torch.empty(B, dtype=torch.int32, device=dev),
                     rates=torch.empty(B, dtype=torch.float32, device=dev),
                     logits=torch.empty(B, dtype=torch.float32, device=dev),
                     infer=torch.empty(B, dtype=torch.float32, device=dev))
            self._stage[key] = b
        return b

    def _capture(self, fn):
        cap = torch.cuda.Stream(device=self.device)
        cap.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(cap):
            check(self.L.tfr_graph_begin_capture(cap.cuda_stream))
            try:
                fn()
            finally:
                exe = C.c_void_p()
                rc = self.L.tfr_graph_end_capture(cap.cuda_stream, C.byref(exe))
            check(rc)
        torch.cuda.current_stream(self.device).wait_stream(cap)
        return exe

    def run_stream_steps(self, n_steps, use_graph=True, pipeline=None):
        """Runs n_steps train steps on batches drawn by the device-resident index stream, starting at the current
        batch_cursor.  With use_graph every step is ONE replay of a captured CUDA graph (no per-step host work
        besides the launch).  With pipeline the graph of step t also assembles and sorts batch t+1 on a side stream
        (two buffer sets, two graphs alternating).  Returns the buffer set of the LAST step (logits / infer of the
        pre-update tables)."""
        B = self.stream_B
        if n_steps <= 0:
            return self.stream_buffers(B, 0)
        if pipeline is None:
            # the forward is fused into the segment sums, which need the sorted ids: sorting the next batch ahead takes
            # the sort off the critical path at every table size
            pipeline = True
        with torch.cuda.device(self.device):
            if not pipeline:
                bufs = self.stream_buffers(B, 0)
                self._primed = None
                if not use_graph:
                    for _ in range(n_steps):
                        self._enqueue_stream_step(B, bufs)
                    return bufs
                g = self._graphs.get((B, "plain"))
                if g is None:
                    self.workspace(B)
                    g = self._graphs[(B, "plain")] = self._capture(lambda: self._enqueue_stream_step(B, bufs))
                st = self._stream()
                for _ in range(n_steps):
                    check(self.L.tfr_graph_launch(g, st))
                return bufs
            return self._run_pipelined(B, n_steps, use_graph, launch=True)

    def prepare_stream_graphs(self, n_steps):
        """Captures (without running anything) every graph run_stream_steps(n_steps) is going to replay from the current
        state, so that no capture / instantiation falls into a timed region."""
        with torch.cuda.device(self.device):
            self._run_pipelined(self.stream_B, n_steps, True, launch=False)

    def _pipe_graph(self, B, slot, K):
        """Graph of K consecutive pipelined steps beginning on buffer set `slot` (K = 1, or an even count so that the
        graph ends on the set it began with)."""
        key = (B, "pipe", slot, K)
        g = self._graphs.get(key)
        if g is None:
            def many():
                for i in range(K):
                    self._enqueue_pipelined_step(B, (slot + i) & 1)
            g = self._graphs[key] = self._capture(many)
        return g

    def _run_pipelined(self, B, n_steps, use_graph, launch):
        for slot in (0, 1):
            self.stream_buffers(B, slot)
            self.workspace((B, slot))
        slot = getattr(self, "_primed", None)
        if slot is None:  # nothing assembled ahead for the batch at the cursor: prime set 0
            slot = 0
            if launch:
                self._prefetch(B, 0, True, self._stream())
        # graphs of `self.graph_steps` consecutive steps: one launch per graph_steps steps instead of one per step --
        # the gap between two graph launches is paid once per graph.  The remainder runs as single-step graphs.
        K = max(2, int(getattr(self, "graph_steps", 8)) // 2 * 2)
        done = 0
        while done < n_steps:
            k = K if (use_graph and n_steps - done >= K) else 1
            if use_graph:
                g = self._pipe_graph(B, slot, k)
                if launch:
                    check(self.L.tfr_graph_launch(g, self._stream()))
            elif launch:
                self._enqueue_pipelined_step(B, slot)
            if k == 1:
                slot = 1 - slot
            done += k
        if launch:
            self._primed = slot  # set `slot` now holds the batch at the (advanced) cursor
        return self.stream_buffers(B, 1 - slot)

    # ---- state access ------------------------------------------------------------------------------------
    def opt_scalars(self):
        raw = self.opt.cpu().numpy().tobytes()
        return OptScalars.from_buffer_copy(raw)

    @property
    def global_step(self):
        return int(self.opt_scalars().global_step)

    def live_slots(self):
        """How many slot-map entries carry the CURRENT step's stamp (0 between steps: a step's entries die when
        global_step advances)."""
        stamp = self.global_step & 0xffffffff
        return sum(int((((m >> 32) & 0xffffffff) == stamp).sum()) for m in (self.user_slot, self.item_slot))

    def get_tables(self):
        out = {n: self.t[n].detach().cpu().numpy().copy() for n in TABLE_NAMES}
        for k, v in self.slots.items():
            out[k] = v.detach().cpu().numpy().copy()
        return out

    def variable(self, name):
        return self.t[name]

    # ---- checkpoint: tf.train.Saver().save / restore (svd_train_val.py:54,197-198; adaptive_test.py:40) -----
    def save(self, path):
        s = self.opt_scalars()
        arrays = self.get_tables()
        arrays["__opt__"] = np.array([s.beta1_power, s.beta2_power], np.float32)
        arrays["__step__"] = np.array([s.global_step], np.int64)
        arrays["__shape__"] = np.array([self.U, self.I, self.d, self.flags], np.int64)
        with open(path, "wb") as f:
            np.savez(f, **arrays)

    @classmethod
    def from_checkpoint(cls, path, device=None):
        """An engine of the shape and model flags recorded in a checkpoint written by save(), restored from it."""
        with np.load(path) as z:
            U, I, d, flags = (int(x) for x in z["__shape__"])
        eng = cls(U, I, d, 1e-3, 0.0, flags=flags, device=device)
        eng.restore(path)
        return eng

    def restore(self, path):
        z = np.load(path)
        U, I, d, _ = (int(x) for x in z["__shape__"])
        if (U, I, d) != (self.U, self.I, self.d):
            raise TfrError("checkpoint shape %s does not match engine %s" % ((U, I, d), (self.U, self.I, self.d)))
        for n in TABLE_NAMES:
            self.t[n].copy_(torch.from_numpy(z[n].reshape(self.t[n].shape)))
            if not self.sgd and ("m_" + n) in z.files:
                self.slots["m_" + n].copy_(torch.from_numpy(z["m_" + n].reshape(self.t[n].shape)))
                self.slots["v_" + n].copy_(torch.from_numpy(z["v_" + n].reshape(self.t[n].shape)))
        self.user_slot.fill_(-1)  # global_step is about to change: stale stamps must not become valid again
        self.item_slot.fill_(-1)
        for field, val, dt in (("beta1_power", z["__opt__"][0], torch.float32), ("beta2_power", z["__opt__"][1], torch.float32),
                               ("global_step", z["__step__"][0], torch.int64)):
            off = getattr(OptScalars, field).offset
            t = torch.tensor([val], dtype=dt).view(torch.uint8)
            self.opt[off:off + t.numel()].copy_(t)
        check(self.L.tfr_svd_begin_step(self.opt.data_ptr(), self._stream()))  # lr_t from the restored beta powers
