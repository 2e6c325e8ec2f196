"""ShardedSvdEngine: the train step with embedding tables + Adam state row-sharded over the ranks of one
NVLink/NVSwitch box (BASELINE configs[4]: 100M users x 10M items, dim 128, 170 GB of state).

Per step, on every rank (one process per GPU, torch.distributed/NCCL for the plumbing):
  1. all-gather of the batch slices' (user, item, rate) -> every rank holds the same global batch   [NCCL, 12 B/rating]
  2. tfr_shard_gather_rows: copy the rows this rank OWNS to their batch positions, zeros elsewhere    [local kernel]
  3. all-reduce(sum) of the [B, dim+1] x 2 gathered buffers: exact (one non-zero term per element) -- every rank
     now has all B user rows and item rows of the batch                                              [NCCL over NVLink]
  4. the single-GPU kernels, unchanged, on LOCAL tables: forward from the gathered rows (identical on all ranks, so
     the error vector and bias_global need no further exchange), sort of the local row keys, ordered segment sums
     (partner rows from the gathered buffers), one Adam pass over the local shard                     [local kernels]
The exchange is ~68 MB per step against a 42.6 GB local table pass at G=8, so scaling is governed by the local pass
(SURVEY 8e).  The reference has no distributed code; this is the B200-native equivalent north_star asks for.

Serving (rank_users, fold_in, rank_folded, similar_items, similar_users) gives the single-GPU results, ids and bits, from
the same sharded tables: query rows (or the rows of the rated items) are gathered to every rank the same way, every rank
ranks its own shard with the single-GPU kernel, and the per-rank lists are all-gathered and merged under the ranking's
total order.
"""
import ctypes as C

import numpy as np
import torch
import torch.distributed as dist

from . import _lib, sharding
from ._lib import ABS_ITEM, LOSS_SIGMOID_CE, OPT_SGD, README_FLAGS, VAR_ALL, OptScalars, SvdTables, TfrError, check
from .engine import FoldedUsers, PairCSR, SvdEngine, check_lengths, csr_of


class ShardedSvdEngine:
    def __init__(self, user_num, item_num, dim, lr, reg, rank, world, flags=README_FLAGS, tables=None, device=None,
                 group=None, device_init_seed=13575):
        """tables: full (unsharded) numpy tables to inject (tests); None -> each rank draws its shard on device.
        Sharded tables train with Adam only, and every rank must own at least one row of each table."""
        self.rank, self.world, self.group = int(rank), int(world), group
        self.U, self.I, self.d = int(user_num), int(item_num), int(dim)
        if int(flags) & OPT_SGD:
            # the SGD slice update would take the "not mine" run for a row, one past the local tables
            raise ValueError("ShardedSvdEngine trains with Adam only: flags %#x include OPT_SGD" % int(flags))
        if min(self.U, self.I) < self.world:
            raise ValueError("ShardedSvdEngine needs at least one row of each table per rank: %d users, %d items, "
                             "world %d" % (self.U, self.I, self.world))
        self.U_loc = sharding.rows_on_rank(self.U, world, rank)
        self.I_loc = sharding.rows_on_rank(self.I, world, rank)
        local = None
        if tables is not None:
            local = dict(mu=tables["mu"], user_bias=sharding.shard_table(tables["user_bias"], world, rank),
                         item_bias=sharding.shard_table(tables["item_bias"], world, rank),
                         user_feat=sharding.shard_table(tables["user_feat"], world, rank),
                         item_feat=sharding.shard_table(tables["item_feat"], world, rank))
        # the local shard is an ordinary engine: same tables struct, same kernels
        self.local = SvdEngine(self.U_loc, self.I_loc, dim, lr, reg, flags=flags, var_mask=VAR_ALL, tables=local,
                               device=device, device_init_seed=device_init_seed + 1000 * rank)
        self.device = self.local.device
        self.L = self.local.L
        self._bufs = {}

    def _buffers(self, B):
        b = self._bufs.get(B)
        if b is None:
            dev, d = self.device, self.d
            # one contiguous exchange buffer: [user rows | item rows | user bias | item bias]
            flat = torch.empty(2 * B * d + 2 * B, dtype=torch.float32, device=dev)
            b = dict(flat=flat, g_uf=flat[:B * d], g_if=flat[B * d:2 * B * d], g_ub=flat[2 * B * d:2 * B * d + B],
                     g_ib=flat[2 * B * d + B:], key_u=torch.empty(B, dtype=torch.int32, device=dev),
                     key_i=torch.empty(B, dtype=torch.int32, device=dev),
                     logits=torch.empty(B, dtype=torch.float32, device=dev),
                     infer=torch.empty(B, dtype=torch.float32, device=dev))
            t = SvdTables()
            C.memmove(C.byref(t), C.byref(self.local.tables_struct), C.sizeof(SvdTables))
            t.g_user_feat, t.g_item_feat = b["g_uf"].data_ptr(), b["g_if"].data_ptr()
            t.g_user_bias, t.g_item_bias = b["g_ub"].data_ptr(), b["g_ib"].data_ptr()
            b["tables"] = t
            self._bufs[B] = b
        return b

    def gather_owned(self, users, items, bufs):
        """Step 2: this rank's half of the row exchange."""
        B, e, st = users.numel(), self.local, self.local._stream()
        check(self.L.tfr_shard_gather_rows(e.t["user_feat"].data_ptr(), e.t["user_bias"].data_ptr(), self.U_loc, self.d,
                                           e.feat_stride,
                                           users.data_ptr(), B, self.world, self.rank, bufs["g_uf"].data_ptr(),
                                           bufs["g_ub"].data_ptr(), bufs["key_u"].data_ptr(), st))
        check(self.L.tfr_shard_gather_rows(e.t["item_feat"].data_ptr(), e.t["item_bias"].data_ptr(), self.I_loc, self.d,
                                           e.feat_stride,
                                           items.data_ptr(), B, self.world, self.rank, bufs["g_if"].data_ptr(),
                                           bufs["g_ib"].data_ptr(), bufs["key_i"].data_ptr(), st))

    def local_step(self, bufs, rates):
        """Step 4: everything after the exchange, on local tables."""
        e = self.local
        B = rates.numel()
        ws = e.workspace(B)
        st = e._stream()
        check(self.L.tfr_svd_begin_step(e.opt.data_ptr(), st))
        check(self.L.tfr_svd_train_step(C.byref(bufs["tables"]), e.opt.data_ptr(), bufs["key_u"].data_ptr(),
                                        bufs["key_i"].data_ptr(), rates.data_ptr(), B, bufs["logits"].data_ptr(),
                                        bufs["infer"].data_ptr(), e.flags, e.var_mask, ws.data_ptr(), ws.numel(), st,
                                        e._side_arr, e._n_side(), e._fj_events))
        return bufs["logits"], bufs["infer"]

    def train_step(self, users, items, rates):
        """users/items/rates: the GLOBAL batch (identical on every rank), device int32/int32/float32 tensors."""
        e = self.local
        users, items, rates = e._dev_i32(users), e._dev_i32(items), e._dev_f32(rates)
        bufs = self._buffers(users.numel())
        with torch.cuda.device(self.device):
            self.gather_owned(users, items, bufs)
            if self.world > 1:
                dist.all_reduce(bufs["flat"], op=dist.ReduceOp.SUM, group=self.group)
            return self.local_step(bufs, rates)

    def train_step_from_slices(self, users_slice, items_slice, rates_slice):
        """Each rank passes ITS slice of the global batch (what its data loader drew); step 1 all-gathers them."""
        e = self.local
        parts = torch.stack([e._dev_i32(users_slice).view(torch.float32), e._dev_i32(items_slice).view(torch.float32),
                             e._dev_f32(rates_slice)])
        if self.world > 1:
            out = torch.empty((self.world,) + tuple(parts.shape), dtype=parts.dtype, device=self.device)
            dist.all_gather_into_tensor(out, parts, group=self.group)
            users = out[:, 0].reshape(-1).view(torch.int32)
            items = out[:, 1].reshape(-1).view(torch.int32)
            rates = out[:, 2].reshape(-1)
        else:
            users, items, rates = parts[0].view(torch.int32), parts[1].view(torch.int32), parts[2]
        return self.train_step(users.contiguous(), items.contiguous(), rates.contiguous())

    # ---- the all-to-all exchange (north_star): ids -> rows back -> gradient records to the owners -----------------------
    # Each rank works on ITS slice of the global batch: B/G forwards, and sorts / sums only the occurrences of rows it
    # owns.  Phases are separate methods so that tests can drive G virtual ranks on one GPU with an emulated exchange;
    # train_step_a2a composes them with torch.distributed (NCCL all_to_all_single with the exact per-peer counts --
    # known on the host a step AHEAD when the next slice is handed over early, so no step waits for a count).
    def _a2a_bufs(self, n):
        key = ("a2a", n)
        b = self._bufs.get(key)
        if b is None:
            dev, G = self.device, self.world
            nb = check(self.L.tfr_shard_bucket_workspace_bytes(n))
            b = dict(ws=torch.empty(nb, dtype=torch.uint8, device=dev), partials=torch.empty(1024, dtype=torch.float32, device=dev),
                     se_partials=torch.empty(1024, dtype=torch.float64, device=dev),
                     sum_err=torch.zeros(1, dtype=torch.float32, device=dev), sum_se=torch.zeros(1, dtype=torch.float64, device=dev))
            self._bufs[key] = b
        return b

    def a2a_bucket(self, users_s, items_s):
        """Phase 1: my slice's ids bucketed by owner.  -> dict(counts [2G] int32 device, send_ids [2n], slot_u, slot_i)."""
        e = self.local
        users_s, items_s = e._dev_i32(users_s), e._dev_i32(items_s)
        n, G, dev = users_s.numel(), self.world, self.device
        b = self._a2a_bufs(n)
        out = dict(n=n, users=users_s, items=items_s, counts=torch.empty(2 * G, dtype=torch.int32, device=dev),
                   send_ids=torch.empty(max(2 * n, 1), dtype=torch.int32, device=dev)[:2 * n],
                   slot_u=torch.empty(max(n, 1), dtype=torch.int32, device=dev)[:n],
                   slot_i=torch.empty(max(n, 1), dtype=torch.int32, device=dev)[:n])
        with torch.cuda.device(dev):
            check(self.L.tfr_shard_bucket(users_s.data_ptr(), items_s.data_ptr(), n, G, out["counts"].data_ptr(),
                                          out["send_ids"].data_ptr(), out["slot_u"].data_ptr(), out["slot_i"].data_ptr(),
                                          b["ws"].data_ptr(), b["ws"].numel(), e._stream()))
        return out

    @staticmethod
    def _i32arr(a):
        a = [int(x) for x in a]
        return (C.c_int32 * max(len(a), 1))(*a)

    def a2a_gather(self, recv_ids, cnt_u, cnt_i):
        """Phase 2 (owner): the rows asked for, as records [row | bias | pad].  cnt_u / cnt_i: per SOURCE rank (host)."""
        total, rs = int(sum(cnt_u) + sum(cnt_i)), self.d + 4
        rec = torch.empty(max(total, 1), rs, dtype=torch.float32, device=self.device)[:total]
        with torch.cuda.device(self.device):
            check(self.L.tfr_shard_gather_records(C.byref(self.local.tables_struct), recv_ids.data_ptr() if total else None,
                                                  self._i32arr(cnt_u), self._i32arr(cnt_i), self.world,
                                                  rec.data_ptr() if total else None, self.local._stream()))
        return rec

    def a2a_forward(self, bk, rec_in, rates_s):
        """Phase 3 (requester): forward + d cost/d logits on my slice; -> (records out [2n, dim+4] = partner row | e,
        logits [n], infer [n], sums2 [2] float64 = my [sum e, sum squared error], to be all-reduced)."""
        e, n, dev, rs = self.local, bk["n"], self.device, self.d + 4
        rates_s = e._dev_f32(rates_s)
        b = self._a2a_bufs(n)
        rec_out = torch.empty(max(2 * n, 1), rs, dtype=torch.float32, device=dev)[:2 * n]
        logits = torch.empty(max(n, 1), dtype=torch.float32, device=dev)[:n]
        infer = torch.empty(max(n, 1), dtype=torch.float32, device=dev)[:n]
        sums2 = torch.empty(2, dtype=torch.float64, device=dev)
        with torch.cuda.device(dev):
            check(self.L.tfr_shard_fwd_records(C.byref(e.tables_struct), e.opt.data_ptr(), rec_in.data_ptr() if n else None,
                                               bk["slot_u"].data_ptr() if n else None, bk["slot_i"].data_ptr() if n else None,
                                               rates_s.data_ptr() if n else None, n, rec_out.data_ptr() if n else None,
                                               logits.data_ptr() if n else None, infer.data_ptr() if n else None,
                                               b["partials"].data_ptr(), b["se_partials"].data_ptr(), sums2.data_ptr(),
                                               e._stream()))
        return rec_out, logits, infer, sums2

    def a2a_owner_step(self, recv_ids, grads_in, cnt_u, cnt_i, sums2, n_slice):
        """Phase 4 (owner): keys + errors by arrival position, then sort -> ordered segment sums -> ONE Adam pass over
        the local shard -> finish (bias_global from the all-reduced sum of e)."""
        e, dev = self.local, self.device
        total = int(sum(cnt_u) + sum(cnt_i))
        cap = 1 << max(10, (max(total, 1) - 1).bit_length())
        ws = e.workspace((cap, "a2a"))
        b = self._a2a_bufs(n_slice)
        carved = _lib.StepWs()
        check(self.L.tfr_svd_step_carve(ws.data_ptr(), ws.numel(), max(total, 1), self.d, C.byref(carved)))
        keys = torch.empty(2, max(total, 1), dtype=torch.int32, device=dev)
        t = SvdTables()
        C.memmove(C.byref(t), C.byref(e.tables_struct), C.sizeof(SvdTables))
        gp = grads_in.data_ptr() if total else None
        t.g_user_feat, t.g_item_feat, t.g_stride = gp, gp, self.d + 4
        with torch.cuda.device(dev):
            st = e._stream()
            check(self.L.tfr_shard_owner_prepare(recv_ids.data_ptr() if total else None, gp, self._i32arr(cnt_u),
                                                 self._i32arr(cnt_i), self.world, self.d, self.U_loc, self.I_loc,
                                                 keys[0].data_ptr(), keys[1].data_ptr(), carved.err, sums2.data_ptr(),
                                                 b["sum_err"].data_ptr(), b["sum_se"].data_ptr(), st))
            check(self.L.tfr_svd_train_step_gathered(C.byref(t), e.opt.data_ptr(), keys[0].data_ptr(), keys[1].data_ptr(),
                                                     total, e.flags, e.var_mask, b["sum_err"].data_ptr(),
                                                     b["sum_se"].data_ptr(), ws.data_ptr(), ws.numel(), st))
        self._keep = (keys, grads_in, recv_ids)   # alive until the stream has consumed them

    def _a2a_plan(self, users_s, items_s):
        """Bucket a slice and exchange the per-peer counts; the counts land in pinned memory behind an event, so a plan
        made a step ahead costs the step that uses it nothing."""
        bk = self.a2a_bucket(users_s, items_s)
        G = self.world
        allc = torch.empty(G, 2 * G, dtype=torch.int32, device=self.device)
        if G > 1:
            dist.all_gather_into_tensor(allc, bk["counts"], group=self.group)
        else:
            allc.copy_(bk["counts"].view(1, -1))
        host = torch.empty(G, 2 * G, dtype=torch.int32).pin_memory()
        host.copy_(allc, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(self.device))
        bk.update(counts_host=host, counts_event=ev, key=(users_s, items_s))
        return bk

    def prepare_slice(self, users_s, items_s):
        """Hand the NEXT step's slice over early (bucket + count exchange on the side stream, under this step's pass)."""
        side = self.local.side_streams[0]
        side.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(side):
            self._plan = self._a2a_plan(users_s, items_s)
        self._plan["side"] = True

    def train_step_a2a(self, users_s, items_s, rates_s, next_slice=None):
        """One step, each rank passing ITS slice of the global batch.  -> (logits, infer) of the slice.  next_slice =
        (users, items) of the FOLLOWING step: bucketed and its counts exchanged under this step's table pass."""
        me, G = self.rank, self.world
        plan = getattr(self, "_plan", None)
        self._plan = None
        if plan is None or plan["key"][0] is not users_s or plan["key"][1] is not items_s:
            plan = self._a2a_plan(users_s, items_s)
        elif plan.get("side"):
            torch.cuda.current_stream(self.device).wait_stream(self.local.side_streams[0])
        plan["counts_event"].synchronize()
        cnt = plan["counts_host"].numpy().astype(np.int64)          # [src, 2G]: users to rank g | items to rank g
        send_cu, send_ci = cnt[me, :G], cnt[me, G:]
        recv_cu, recv_ci = cnt[:, me], cnt[:, G + me]
        send_splits, recv_splits = (send_cu + send_ci).tolist(), (recv_cu + recv_ci).tolist()
        total, n, rs, dev = int(sum(recv_splits)), plan["n"], self.d + 4, self.device
        recv_ids = torch.empty(max(total, 1), dtype=torch.int32, device=dev)[:total]
        rec_in = torch.empty(max(2 * n, 1), rs, dtype=torch.float32, device=dev)[:2 * n]
        grads_in = torch.empty(max(total, 1), rs, dtype=torch.float32, device=dev)[:total]
        if G > 1:
            dist.all_to_all_single(recv_ids, plan["send_ids"], recv_splits, send_splits, group=self.group)
        else:
            recv_ids.copy_(plan["send_ids"])
        rec = self.a2a_gather(recv_ids, recv_cu, recv_ci)
        if G > 1:
            dist.all_to_all_single(rec_in, rec, send_splits, recv_splits, group=self.group)
        else:
            rec_in.copy_(rec)
        rec_out, logits, infer, sums2 = self.a2a_forward(plan, rec_in, rates_s)
        if G > 1:
            dist.all_reduce(sums2, op=dist.ReduceOp.SUM, group=self.group)
            dist.all_to_all_single(grads_in, rec_out, recv_splits, send_splits, group=self.group)
        else:
            grads_in.copy_(rec_out)
        if next_slice is not None:
            self.prepare_slice(*next_slice)
        self.a2a_owner_step(recv_ids, grads_in, recv_cu, recv_ci, sums2, n)
        return logits, infer

    def a2a_exchange_bytes(self, B):
        """Bytes this rank SENDS per step in the three all-to-alls (ids, rows back, gradient records), on average."""
        n = B // self.world
        return 2 * n * 4 + 2 * 2 * n * (self.d + 4) * 4

    def exchange_bytes(self, B):
        """Bytes this rank contributes to the per-step collectives (ids all-gather + rows all-reduce)."""
        return 12 * (B // self.world) + 4 * (2 * B * self.d + 2 * B)

    def get_local_tables(self):
        return self.local.get_tables()

    # ---- serving: exact top-k and fold-in from the sharded tables ---------------------------------------------------------
    # Collective calls: every rank passes the same arguments and gets the same result, the ids and bits SvdEngine gives on
    # the re-assembled tables.  Ids are checked against the global tables on every rank before any collective, so every
    # rank raises together.  The phases (gather / exclusion lists / local rank / merge) are separate methods so that tests
    # can drive G virtual ranks on one GPU with the collectives emulated; the public methods compose them with
    # torch.distributed, or with nothing at world 1.
    def _check_ids(self, users, items, n_users=None):
        SvdEngine._check_ids(self, users, items, n_users)   # against the GLOBAL U and I

    def _dev_i32(self, a):
        return self.local._dev_i32(a)

    def _dev_f32(self, a):
        return self.local._dev_f32(a)

    def _all_reduce(self, t):
        if self.world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group)
        return t

    def _all_gather(self, t):
        """[G, *t.shape]: every rank's t, by rank (all_gather_into_tensor)."""
        if self.world == 1:
            return t.unsqueeze(0)
        out = torch.empty((self.world,) + tuple(t.shape), dtype=t.dtype, device=self.device)
        dist.all_gather_into_tensor(out, t.contiguous(), group=self.group)
        return out

    def _gather_rows(self, feat, bias, rows_local, ids):
        """tfr_shard_gather_rows of a local table: the rows of ids (device int32, global) this rank owns at their
        positions, zeros elsewhere, as one buffer [m rows of d | m biases]; summed over the ranks it holds every row.
        An all-reduce adds the +0.0 of the ranks that do not own a row, so an owned -0.0 arrives as +0.0.  No result bit
        depends on that: the scorer's dot product and the fold-in Gram and right-hand side are float64 sums that start
        from +0.0, a product with a zero factor is a zero, and in round-to-nearest +0.0 + (-0.0) = +0.0 + (+0.0) = +0.0,
        so such a sum is never -0.0 and adding either zero to it (or a bias, or mu, after it) gives the same bits.  The
        norms of similar_items / similar_users are such sums too: the square of either zero is +0.0."""
        m, d, e = ids.numel(), self.d, self.local
        flat = torch.empty(max(m * d + m, 1), dtype=torch.float32, device=self.device)
        keys = torch.empty(max(m, 1), dtype=torch.int32, device=self.device)
        check(self.L.tfr_shard_gather_rows(feat.data_ptr(), bias.data_ptr(), rows_local, d, e.feat_stride, ids.data_ptr(),
                                           m, self.world, self.rank, flat.data_ptr(), flat[m * d:].data_ptr(),
                                           keys.data_ptr(), e._stream()))
        return flat

    def pair_csr(self, users, items):
        """An exclusion set for rank_users from GLOBAL (user, item) pairs, built once per training set: this rank's share,
        the distinct pairs whose item it owns, as a PairCSR by global user id with global item ids.  Not collective."""
        self._check_ids(users, items)
        u, i = self._dev_i32(users).to(torch.int64), self._dev_i32(items).to(torch.int64)
        keep = i % self.world == self.rank
        key = torch.unique(u[keep] * self.I + i[keep])   # sorted
        indptr, items, _ = csr_of(key // self.I, key % self.I, self.U, self.I)
        return PairCSR(indptr, items)

    def serve_gather(self, q):
        """Phase 1 of rank_users: the query users' rows (q device int32, global ids) this rank owns; summed over the ranks
        (all-reduce) the buffer is the n-row user table [n rows of d | n biases] of the queries, row j = user q[j]."""
        with torch.cuda.device(self.device):
            return self._gather_rows(self.local.t["user_feat"], self.local.t["user_bias"], self.U_loc, q)

    def serve_exclusions(self, csr, rows):
        """This rank's exclusion lists by query position: the items of csr's rows `rows` (device int32) that it owns, as
        ascending local ids -- a PairCSR over len(rows) rows (tfr_shard_excl_indptr / _fill; one total read back)."""
        n, dev = rows.numel(), self.device
        indptr = torch.empty(n + 1, dtype=torch.int64, device=dev)
        nbytes = check(self.L.tfr_shard_excl_workspace_bytes(n))
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        args = (csr.indptr.data_ptr(), csr.items.data_ptr(), csr.indptr.numel() - 1, rows.data_ptr(), n, self.world,
                self.rank)
        with torch.cuda.device(dev):
            st = self.local._stream()
            check(self.L.tfr_shard_excl_indptr(*args, indptr.data_ptr(), ws.data_ptr(), nbytes, st))
            items = torch.empty(int(indptr[n]), dtype=torch.int32, device=dev)
            check(self.L.tfr_shard_excl_fill(*args, indptr.data_ptr(), items.data_ptr(), st))
        return PairCSR(indptr, items)

    def serve_rank(self, user_feat, user_bias, k, excl):
        """Phase 2: tfr_rank_users of every row of an n-row user table (the gathered queries, or folded users) against
        this rank's item shard -> (local item ids [n, k], scores [n, k]).  k: of the WHOLE item table, so that every
        rank's list has the same shape (a shard with fewer items pads with (-inf, -1)); excl: serve_exclusions or None."""
        n = int(user_bias.numel())
        q = torch.arange(n, dtype=torch.int32, device=self.device)
        return self.local._rank_rows(user_feat, user_bias, n, 0, q, k, excl)

    def serve_merge(self, val, idx):
        """Phase 3: the all-gathered lists val / idx [G, n, k] -> (items [n, k] int32 global ids, scores [n, k] float64),
        the top k of their union (tfr_shard_topk_merge)."""
        G, n, k = idx.shape
        if G != self.world:
            raise TfrError("serve_merge: %d lists for a world of %d" % (G, self.world))
        out_idx = torch.empty(n, k, dtype=torch.int32, device=self.device)
        out_val = torch.empty(n, k, dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            check(self.L.tfr_shard_topk_merge(val.data_ptr(), idx.data_ptr(), G, n, k, out_val.data_ptr(),
                                              out_idx.data_ptr(), self.local._stream()))
        return out_idx, out_val

    def _rank_table(self, user_feat, user_bias, k, excl):
        idx, val = self.serve_rank(user_feat, user_bias, k, excl)
        return self.serve_merge(self._all_gather(val), self._all_gather(idx))

    def rank_users(self, users, k=50, exclude=None):
        """SvdEngine.rank_users on the sharded model: -> (items [n, k] int32 global ids, scores [n, k] float64) on the
        device, identical in ids and bits to SvdEngine.rank_users on the re-assembled tables with the same exclude.
        exclude: global (users, items) pairs, or a PairCSR from pair_csr() (build it once).  Collective: the query rows
        are gathered to every rank, each ranks its item shard, and the per-rank lists are all-gathered and merged."""
        self._check_ids(users, [])
        csr = None
        if exclude is not None:
            csr = exclude if isinstance(exclude, PairCSR) else self.pair_csr(*exclude)
        q = self._dev_i32(np.atleast_1d(np.asarray(users)) if not isinstance(users, torch.Tensor) else users.reshape(-1))
        n, d, k = q.numel(), self.d, int(min(k, self.I))
        if n == 0:
            return (torch.empty(0, k, dtype=torch.int32, device=self.device),
                    torch.empty(0, k, dtype=torch.float64, device=self.device))
        with torch.cuda.device(self.device):
            table = self._all_reduce(self.serve_gather(q))
            excl = self.serve_exclusions(csr, q) if csr is not None else None
            return self._rank_table(table[:n * d].view(n, d), table[n * d:n * d + n], k, excl)

    def fold_gather(self, ids):
        """Phase 1 of fold_in: the rows of the rated items ids (device int32, distinct, ascending) this rank owns; summed
        over the ranks (all-reduce) the buffer is the compact item table [m rows of d | m biases], row j = item ids[j]."""
        with torch.cuda.device(self.device):
            return self._gather_rows(self.local.t["item_feat"], self.local.t["item_bias"], self.I_loc, ids)

    def fold_plan(self, rows, items, rates, n=None, reg=None):
        """Phase 0 of fold_in, the same on every rank: the refusals of SvdEngine.fold_in, the ratings CSR as SvdEngine
        builds it (global ids), the distinct rated items (ascending) and each rating's position among them."""
        e = self.local
        if e.flags & LOSS_SIGMOID_CE:
            raise TfrError("fold_in solves the squared-error objective; the sigmoid cross-entropy model is not supported")
        reg = e.hyper["reg"] if reg is None else float(reg)
        if not reg >= 0.0:
            raise TfrError("fold_in: reg must be >= 0, got %r" % reg)
        size = check_lengths("fold_in", "rows, items and rates", rows, items, rates)
        if n is None:
            n = int((rows if isinstance(rows, torch.Tensor) else np.asarray(rows)).max()) + 1 if size else 0
        n = int(n)
        indptr, it, rt = SvdEngine._csr_by_user(self, rows, items, rates, n_rows=n)   # checks ids against n and I
        ids, pos = torch.unique(it, return_inverse=True)   # sorted: positions keep the CSR's order
        return dict(n=n, reg=reg, indptr=indptr, items=it, rates=rt, ids=ids.to(torch.int32).contiguous(),
                    pos=pos.to(torch.int32).contiguous())

    def fold_gather(self, ids):
        """Phase 1 of fold_in: the rows of the rated items ids (device int32, global) this rank owns; summed over the
        ranks (all-reduce) the buffer is the compact item table [m rows of d | m biases], row j = item ids[j]."""
        with torch.cuda.device(self.device):
            return self._gather_rows(self.local.t["item_feat"], self.local.t["item_bias"], self.I_loc, ids)

    def fold_solve(self, plan, table):
        """Phase 2 of fold_in: tfr_fold_in_users against the compact item table, ratings by position in it."""
        e, dev, d, n, m = self.local, self.device, self.d, plan["n"], plan["ids"].numel()
        feat = torch.empty(n, d, dtype=torch.float32, device=dev)
        bias = torch.empty(n, dtype=torch.float32, device=dev)
        info = torch.empty(n, dtype=torch.int32, device=dev)
        with torch.cuda.device(dev):
            check(self.L.tfr_fold_in_users(table.data_ptr(), table[m * d:].data_ptr(), e.t["mu"].data_ptr(), m, d, 0,
                                           e.flags, plan["reg"], plan["indptr"].data_ptr(), plan["pos"].data_ptr(),
                                           plan["rates"].data_ptr(), n, feat.data_ptr(), bias.data_ptr(), info.data_ptr(),
                                           e._stream()))
        return FoldedUsers(feat, bias, PairCSR(plan["indptr"], plan["items"]), info)

    def fold_in(self, rows, items, rates, n=None, reg=None):
        """SvdEngine.fold_in on the sharded item side, the same FoldedUsers in bits (feat, bias, info; ratings with global
        item ids).  Collective: the rows of the distinct rated items are gathered to every rank as a compact table, the
        ratings CSR is built as SvdEngine builds it and its ids replaced by positions in that table, and every rank
        solves the same systems (tfr_fold_in_users): tiny, redundant work that needs no broadcast.  Refuses what
        SvdEngine.fold_in refuses, with TfrError."""
        plan = self.fold_plan(rows, items, rates, n, reg)
        return self.fold_solve(plan, self._all_reduce(self.fold_gather(plan["ids"])))

    def similar_gather(self, q, items):
        """Phase 1 of similar_items / similar_users: the query rows (q device int32, global ids) this rank owns; summed over
        the ranks (all-reduce) the buffer is the n-row table of the queries [n rows of d | n biases], row j = row q[j]
        (items: the gather of fold_gather; users: the gather of serve_gather)."""
        return self.fold_gather(q) if items else self.serve_gather(q)

    def similar_rank(self, table, q, k, items):
        """Phase 2: tfr_similar_rows of every gathered query row (table: similar_gather's buffer, all-reduced) against this
        rank's shard of the same table -> (local ids [n, k], scores [n, k]).  The query's own row is skipped where this
        rank owns it (local id q // G).  k: of the WHOLE table, so that every rank's list has the same shape."""
        e, n, G = self.local, int(q.numel()), self.world
        qi = q.to(torch.int64)
        skip = torch.where(qi % G == self.rank, qi // G, -1).to(torch.int32).contiguous()
        rows = torch.arange(n, dtype=torch.int32, device=self.device)
        feat, n_loc = (e.t["item_feat"], self.I_loc) if items else (e.t["user_feat"], self.U_loc)
        abs_rows = items and bool(e.flags & ABS_ITEM)
        return e._similar_rows(table[:n * self.d], n, 0, rows, skip, feat, n_loc, abs_rows, k)

    def _similar(self, ids, k, items):
        if items:
            self._check_ids([], ids)
        else:
            self._check_ids(ids, [])
        q = self._dev_i32(np.atleast_1d(np.asarray(ids)) if not isinstance(ids, torch.Tensor) else ids.reshape(-1))
        n, k = q.numel(), int(min(k, self.I if items else self.U))
        if n == 0:
            return (torch.empty(0, k, dtype=torch.int32, device=self.device),
                    torch.empty(0, k, dtype=torch.float64, device=self.device))
        with torch.cuda.device(self.device):
            idx, val = self.similar_rank(self._all_reduce(self.similar_gather(q, items)), q, k, items)
            return self.serve_merge(self._all_gather(val), self._all_gather(idx))

    def similar_items(self, items, k=10):
        """SvdEngine.similar_items on the sharded model: the same ids and bits as on the re-assembled tables.  Collective:
        the query rows are gathered to every rank, each ranks its own item shard by cosine, and the per-rank lists are
        all-gathered and merged (tfr_shard_topk_merge)."""
        return self._similar(items, k, True)

    def similar_users(self, users, k=10):
        """SvdEngine.similar_users on the sharded model, as similar_items.  Collective."""
        return self._similar(users, k, False)

    def rank_folded(self, folded, k=50, exclude_rated=True):
        """SvdEngine.rank_folded on the sharded item side, the same ids and bits.  The folded rows are on every rank
        already (fold_in solves them everywhere): each rank ranks its item shard, the lists are all-gathered and merged.
        exclude_rated: never recommend the items the row was folded in from.  Collective."""
        n, k = int(folded.feat.shape[0]), int(min(k, self.I))
        if n == 0:
            return (torch.empty(0, k, dtype=torch.int32, device=self.device),
                    torch.empty(0, k, dtype=torch.float64, device=self.device))
        with torch.cuda.device(self.device):
            excl = None
            if exclude_rated:
                excl = self.serve_exclusions(folded.ratings, torch.arange(n, dtype=torch.int32, device=self.device))
            return self._rank_table(folded.feat, folded.bias, k, excl)
