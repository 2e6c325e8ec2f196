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
"""
import ctypes as C

import numpy as np
import torch
import torch.distributed as dist

from . import _lib, sharding
from ._lib import OPT_SGD, README_FLAGS, VAR_ALL, OptScalars, SvdTables, check
from .engine import SvdEngine


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
