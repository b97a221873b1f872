"""Model classes with the reference's interface (models/sasrec.py:5,127; models/cast_1.py:6,158 ...).

    model = SASRec(usernum, itemnum, args)            # or CAST1..CAST9(usernum, itemnum, ratingnum, args)
    auc, loss = model.train_step(u, seq, pos, neg, time_seq, hours, days)      # == sess.run([auc, loss, train_op])
    logits, attn = model.predict(sess, u, seq, item_idx, timeseq=..., hours_seq=..., days_seq=...)

`args` is the reference's argparse namespace (main.py:42-86); `sess` is accepted and ignored.  Inputs are host
numpy int arrays as produced by the reference's sampler; results are host floats / numpy arrays.
"""
from __future__ import annotations

from typing import Optional

import numpy as np
import torch

from .engine import Engine, MODELS


class _Model:
    registry_name = "sasrec"

    def __init__(self, usernum, itemnum, args, *, device=None, use_graph: bool = True, _lib=None, seed=None,
                 item_shard=None, alloc=None):
        self.usernum, self.itemnum, self.args = usernum, itemnum, args
        self.engine = Engine(self.registry_name, usernum, itemnum, args, device=device, lib=_lib, seed=seed,
                             item_shard=item_shard, alloc=alloc)
        self.use_graph = bool(use_graph) and self.engine.device.type == "cuda"
        self.attention_weights = None
        self.launches_per_step = None
        self._pinned = {}
        self._sums_host = None

    # ------------------------------------------------------------------ helpers
    def use_device_time_features(self, bin_in_hours=48, max_bins=200, log_scale=False, min_timedelta=None,
                                 max_timedelta=None):
        """Derive the time-bin / hour / weekday ids on the device from raw int64 timestamps (`timestamps=` of
        train_step / predict / score_candidates) with the dataset's bin rule — reference util.py:24-43,73-120 applied
        per position by sampler.py:61-72 and util.py:276-289."""
        from .timefeat import TimeFeaturizer
        eng = self.engine
        self.timefeat = TimeFeaturizer(eng.device, bin_in_hours, max_bins, log_scale, min_timedelta, max_timedelta,
                                       lib=eng.lib)
        return self

    def _stage_timestamps(self, c, timestamps):
        """raw timestamps -> c.cids on the device (after the item ids of the batch are staged)"""
        eng = self.engine
        if getattr(self, "timefeat", None) is None:
            raise ValueError("timestamps= needs use_device_time_features(...) first (the dataset's bin rule)")
        B, T = c.B, eng.T
        key = (B, "ts")
        st = self._pinned.get(key)
        if st is None:
            pin = eng.device.type == "cuda"
            host = torch.zeros(B, T, dtype=torch.int64, pin_memory=pin)
            st = self._pinned[key] = {"host": host, "hostn": host.numpy(),
                                      "dev": torch.zeros(B, T, dtype=torch.int64, device=eng.device), "event": None}
        if st["event"] is not None:
            st["event"].synchronize()
        np.copyto(st["hostn"], np.asarray(timestamps).reshape(B, T), casting="unsafe")
        st["dev"].copy_(st["host"], non_blocking=True)
        if eng.device.type == "cuda":
            st["event"] = torch.cuda.Event()
            st["event"].record(torch.cuda.current_stream(eng.device))
        self.timefeat.into(st["dev"], c.keys3[0], c.cids)

    def _stage(self, c, seq, pos, neg, time_seq, hours, days):
        """host -> device copies of one batch into the static input buffers: pinned staging, non-blocking copies.
        Three staging sets rotate and each remembers the event recorded after its copies, so `train_step_async` can be
        called back to back without a batch being overwritten before its copy has run."""
        eng = self.engine
        B, T = c.B, eng.T
        key = (B, "in")
        ring = self._pinned.get(key)
        if ring is None:
            pin = eng.device.type == "cuda"
            ring = {"slots": [], "next": 0}
            for _ in range(3 if pin else 1):
                k3 = torch.zeros(3, B * T, dtype=torch.int32, pin_memory=pin)
                c3 = torch.zeros(3, B * T, dtype=torch.int32, pin_memory=pin)
                # numpy views of the pinned buffers: np.copyto has far less overhead than Tensor.copy_
                ring["slots"].append({"k3": k3, "c3": c3, "k3n": k3.numpy(), "c3n": c3.numpy(), "event": None})
            self._pinned[key] = ring
        st = ring["slots"][ring["next"]]
        ring["next"] = (ring["next"] + 1) % len(ring["slots"])
        if st["event"] is not None:
            st["event"].synchronize()       # the copy that last used this slot has completed
        k3n, c3n = st["k3n"], st["c3n"]
        for j, a in enumerate((seq, pos, neg)):
            if a is not None:
                np.copyto(k3n[j], np.asarray(a).reshape(-1), casting="unsafe")
            else:
                k3n[j].fill(0)
        c.keys3.copy_(st["k3"], non_blocking=True)
        tables = eng.plan.tables
        need = [("time_emb", time_seq), ("hours_emb", hours), ("days_emb", days)]
        if any(t in tables for t, _ in need):
            if all(a is None for _, a in need) and getattr(self, "_ts_pending", None) is not None:
                return      # raw timestamps follow: the device fills c.cids (_stage_timestamps)
            for j, (t, a) in enumerate(need):
                if t in tables:
                    if a is None:
                        raise ValueError(f"model {self.registry_name} needs the {t[:-4]} sequence")
                    np.copyto(c3n[j], np.asarray(a).reshape(-1), casting="unsafe")
            c.cids.copy_(st["c3"], non_blocking=True)
        if eng.device.type == "cuda":
            st["event"] = torch.cuda.Event()
            st["event"].record(torch.cuda.current_stream(eng.device))

    def _capture(self, c):
        """Capture the step as CUDA graphs: [forward+loss+backward] and [Adam]; under data parallelism the NCCL
        all-reduce runs between the two replays (3 host launches per step instead of ~70)."""
        eng = self.engine
        # one eager step first (lazy CUDA init, smem attributes), with parameters / optimizer state restored after
        saved = (eng.w.clone(), eng.m.clone(), eng.v.clone(), eng.adam_state.clone())
        n0 = eng.lib.cast_launch_count()
        eng.launch_train_step(c)
        self.launches_per_step = int(eng.lib.cast_launch_count() - n0)
        torch.cuda.synchronize(eng.device)
        eng.w.copy_(saved[0]); eng.m.copy_(saved[1]); eng.v.copy_(saved[2]); eng.adam_state.copy_(saved[3])
        s = torch.cuda.Stream(device=eng.device)
        s.wait_stream(torch.cuda.current_stream(eng.device))
        g1, g2 = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
        # one process, or an exchange made of kernel launches only (dist.PeerExchange): the whole step is one graph
        single = (eng.grad_allreduce is None and eng.after_adam is None) or eng.exchange_capturable
        with torch.cuda.stream(s):
            with torch.cuda.graph(g1, stream=s):
                eng.launch_fwd_bwd(c)
                if single:
                    if eng.grad_allreduce is not None:
                        eng.grad_allreduce(c)
                    eng.adam(c)
                    if eng.after_adam is not None:
                        eng.after_adam()
            if not single:
                with torch.cuda.graph(g2, stream=s):
                    eng.adam(c)
            else:
                g2 = None
        torch.cuda.current_stream(eng.device).wait_stream(s)
        eng.w.copy_(saved[0]); eng.m.copy_(saved[1]); eng.v.copy_(saved[2]); eng.adam_state.copy_(saved[3])
        c.graph = (g1, g2)

    def launch(self, c):
        """Enqueue one training step on the batch already resident in c.keys3 / c.cids."""
        eng = self.engine
        if self.use_graph:
            if c.graph is None:
                self._capture(c)
            c.graph[0].replay()
            if c.graph[1] is not None:
                if eng.grad_allreduce is not None:
                    eng.grad_allreduce(c)
                c.graph[1].replay()
                if eng.after_adam is not None:
                    eng.after_adam()
        else:
            eng.launch_train_step(c)

    def _score_cand(self, last, ld, B, cand, Cn, logits, cgt=None, ceq=None):
        """logits (+ rank counts) of per-user candidate lists; the item rows come from the local table or, with a
        row-sharded table, from the owning ranks' shards"""
        eng = self.engine
        p = eng._p
        if eng.item_shard is not None:
            eng._call(eng.lib.cast_score_rank_cand_sharded, last.data_ptr(), ld, eng.shard_ptrs.data_ptr(),
                      eng.item_shard[1], eng.V_items, eng.H, B, cand.data_ptr(), Cn, logits.data_ptr(), p(cgt), p(ceq),
                      eng._stream())
        else:
            eng._call(eng.lib.cast_score_rank_cand, last.data_ptr(), ld, eng.P["item_emb"].data_ptr(),
                      eng.P["item_emb"].shape[0], eng.H, B, cand.data_ptr(), Cn, logits.data_ptr(), p(cgt), p(ceq),
                      eng._stream())

    def _id_csr(self, lists, n, local_rows=False):
        """Per-user id collections -> CSR device tensors (ptr [n+1], idx), ids unique and ascending per user.
        local_rows=True (row-sharded table): keeps the ids this rank's shard holds, as local rows (id // n_ranks, +1 on
        ranks > 0) — the map is increasing, so each row stays ascending."""
        eng = self.engine
        ptr = np.zeros(n + 1, np.int32)
        flat = []
        for u, r in enumerate(lists):
            ids = np.unique(np.asarray(list(r), dtype=np.int64))
            if local_rows:
                rank, world = eng.item_shard
                ids = ids[(ids % world == rank) & (ids > 0) & (ids < eng.V_items)] // world + (1 if rank else 0)
            flat.append(ids)
            ptr[u + 1] = ptr[u] + len(ids)
        idx = np.concatenate(flat + [np.zeros(1, np.int64)]).astype(np.int32)
        return torch.from_numpy(ptr).to(eng.device), torch.from_numpy(idx).to(eng.device)

    def _topk(self, last, ld, U, V, k, eptr, eidx, mode):
        """cast_topk_full over the rows [0, V) of this process's item table; (ids, scores) [U, k] device tensors"""
        import ctypes
        eng = self.engine
        dev = eng.device
        table = eng.P["item_emb"]
        ids = torch.empty(U, k, dtype=torch.int32, device=dev)
        scores = torch.empty(U, k, dtype=torch.float32, device=dev)
        wsb = eng.lib.cast_topk_full_workspace_bytes(U, V, eng.H, k)
        ws = self._pinned.get("tkws")     # one buffer, grown on demand (the operand images of a large catalog are GBs)
        if ws is None or ws.numel() * 4 < wsb:
            self._pinned["tkws"] = None
            ws = self._pinned["tkws"] = torch.empty(wsb // 4 + 16, dtype=torch.int32, device=dev)
        eng._call(eng.lib.cast_topk_full, last.data_ptr(), ld, table.data_ptr(), V, eng.H, U, k, eng._p(eptr),
                  eng._p(eidx), mode, ids.data_ptr(), scores.data_ptr(), None, ws.data_ptr(), wsb, eng._stream())
        if mode == 0:
            flag = ctypes.c_int(0)
            eng._call(eng.lib.cast_topk_full_status, ws.data_ptr(), U, V, eng.H, k, ctypes.byref(flag), eng._stream())
            if flag.value != 0:
                raise RuntimeError("topk_full: tensor-core pass watchdog fired")
        return ids, scores

    def recommend(self, seq, k=10, exclude=None, time_seq=None, hours=None, days=None, timestamps=None, mode: int = 0):
        """Exact top-k recommendation from the last position of each sequence: the k items of [1, itemnum] not in
        exclude[u] (optional, one id collection per user) with the largest canonical fp32 logits (the logits of
        score_candidates / predict), ties broken by item id ascending.  mode 0 = tcgen05 tensor cores as an exact
        filter, mode 1 = exact brute force; both return the same bits.  Returns (ids [U,k] int32, scores [U,k] float32);
        fewer than k eligible items pad the tail with id 0 and score -inf.  With a row-sharded item table this is a
        collective call (every rank passes its own users, the same count on every rank)."""
        eng = self.engine
        if eng.item_shard is not None:
            return self._recommend_sharded(seq, k, exclude, time_seq, hours, days, timestamps, mode)
        c = self.forward_eval(seq, time_seq, hours, days, timestamps=timestamps)
        B, T, H = c.B, eng.T, eng.H
        eptr, eidx = self._id_csr(exclude, B) if exclude is not None else (None, None)
        last = c.seq_emb.view(B, T, H)[:, T - 1, :]
        ids, scores = self._topk(last, T * H, B, eng.P["item_emb"].shape[0], k, eptr, eidx, mode)
        return ids.cpu().numpy(), scores.cpu().numpy()

    def _recommend_sharded(self, seq, k, exclude, time_seq, hours, days, timestamps, mode):
        """Top-k with the item table sharded by row: the last-position vectors of all ranks are all-gathered, each rank
        takes the top k of its own shard (local rows -> global ids, an increasing map, so the tie order holds), the
        [U, k] lists are all-gathered and merged per user by (score desc, id asc)."""
        import torch.distributed as dist
        eng = self.engine
        rank, world = eng.item_shard
        dev = eng.device
        c = self.forward_eval(seq, time_seq, hours, days, timestamps=timestamps)
        B, T, H = c.B, eng.T, eng.H
        last = c.seq_emb.view(B, T, H)[:, T - 1, :].contiguous()
        U = B * world
        last_all = torch.empty(U, H, dtype=torch.float32, device=dev)
        dist.all_gather_into_tensor(last_all, last)
        excl_all = [None] * world
        dist.all_gather_object(excl_all, None if exclude is None else [sorted(set(int(i) for i in r)) for r in exclude])
        off = 1 if rank else 0
        v_loc = (eng.V_items - rank + world - 1) // world + off      # rows of this shard that hold items (+ the pad)
        ids = torch.zeros(U, k, dtype=torch.int32, device=dev)
        scores = torch.full((U, k), float("-inf"), dtype=torch.float32, device=dev)
        if v_loc > 1:
            eptr = eidx = None
            if excl_all[0] is not None:
                eptr, eidx = self._id_csr([r for rl in excl_all for r in rl], U, local_rows=True)
            rows, scores = self._topk(last_all, H, U, v_loc, k, eptr, eidx, mode)
            ids = torch.where(rows > 0, (rows - off) * world + rank, rows)
        parts_i = [torch.empty_like(ids) for _ in range(world)]
        parts_s = [torch.empty_like(scores) for _ in range(world)]
        dist.all_gather(parts_i, ids)
        dist.all_gather(parts_s, scores)
        all_i = np.concatenate([t.cpu().numpy() for t in parts_i], 1)
        all_s = np.concatenate([t.cpu().numpy() for t in parts_s], 1)
        order = np.lexsort((all_i, -all_s), axis=-1)[:, :k]
        mine = slice(rank * B, (rank + 1) * B)
        return np.take_along_axis(all_i, order, 1)[mine], np.take_along_axis(all_s, order, 1)[mine]

    # ------------------------------------------------------------------ reference protocol
    def _stage_all(self, c, seq, pos, neg, time_seq, hours, days, timestamps):
        self._ts_pending = timestamps if len(self.engine.plan.tables) > 1 else None
        try:
            self._stage(c, seq, pos, neg, time_seq, hours, days)
            if self._ts_pending is not None:
                self._stage_timestamps(c, timestamps)
        finally:
            self._ts_pending = None

    def train_step_async(self, u, seq, pos, neg, time_seq=None, hours=None, days=None, timestamps=None):
        """Enqueue one training step; returns the device tensor {sum loss terms, sum auc terms, sum istarget}.
        timestamps (raw int64 [B,T], 0 = padding) replaces time_seq / hours / days: see use_device_time_features."""
        eng = self.engine
        seq = np.asarray(seq)
        B = seq.shape[0]
        c = eng.ctx(B)
        self._stage_all(c, seq, pos, neg, time_seq, hours, days, timestamps)
        self.launch(c)
        return eng.global_sums()

    def train_step(self, u, seq, pos, neg, time_seq=None, hours=None, days=None, timestamps=None, sync=True):
        """== sess.run([model.auc, model.loss, model.train_op], feed) of reference main.py:212-219.
        sync=False (a training loop that only logs now and then, like the reference's once-per-epoch print): the step's
        {loss, auc, count} sums are still copied to pinned host memory, but the call returns without waiting for them —
        it hands back the (auc, loss) of the PREVIOUS step (None on the first call), so the host prepares batch i+1
        while the GPU runs step i.  `last_metrics()` waits for and returns the newest step's values."""
        s = self.train_step_async(u, seq, pos, neg, time_seq, hours, days, timestamps)
        if s.device.type != "cuda":
            loss_sum, auc_sum, cnt = s[:3].tolist()
            self._lag = None
            self._lag_cpu = (auc_sum / cnt, loss_sum / cnt)
            return self._lag_cpu
        if self._sums_host is None:   # 12-byte read-backs into two alternating pinned slots
            self._sums_host = torch.zeros(2, 4, dtype=torch.float32, pin_memory=True)
            self._sums_ev = [torch.cuda.Event(), torch.cuda.Event()]
            self._lag = None
            self._sums_i = 0
        slot = self._sums_i & 1
        self._sums_i += 1
        prev, self._lag = self._lag, slot
        self._sums_host[slot].copy_(s[:4], non_blocking=True)
        self._sums_ev[slot].record(torch.cuda.current_stream(s.device))
        if sync:
            return self.last_metrics()
        return self._read_metrics(prev) if prev is not None else None

    def _read_metrics(self, slot):
        self._sums_ev[slot].synchronize()
        loss_sum, auc_sum, cnt = self._sums_host[slot][:3].tolist()
        return auc_sum / cnt, loss_sum / cnt

    def last_metrics(self):
        """(auc, loss) of the most recent train_step call (waits for it)."""
        if getattr(self, "_lag", None) is None:
            return getattr(self, "_lag_cpu", None)
        return self._read_metrics(self._lag)

    def forward_eval(self, seq, time_seq=None, hours=None, days=None, want_attn=False, timestamps=None):
        """is_training=False forward; returns the device buffer seq_emb [B*T, H] (and fills attention weights)."""
        eng = self.engine
        seq = np.asarray(seq)
        B = seq.shape[0]
        c = eng.ctx(B)
        self._stage_all(c, seq, None, None, time_seq, hours, days, timestamps)
        eng.forward(c, train=False, want_attn=want_attn)
        return c

    def predict(self, sess, u, seq, item_idx, timeseq=None, input_context_seq=None, hours_seq=None, days_seq=None,
                timestamps=None):
        """reference models/sasrec.py:127-129 / cast_3.py:191-194: returns [test_logits [B,101], attention_weights]."""
        eng = self.engine
        c = self.forward_eval(seq, timeseq, hours_seq, days_seq, want_attn=True, timestamps=timestamps)
        B, T, H = c.B, eng.T, eng.H
        item_idx = np.asarray(item_idx, dtype=np.int32).reshape(-1)
        Cn = item_idx.shape[0]
        cand = torch.from_numpy(np.ascontiguousarray(np.broadcast_to(item_idx, (B, Cn)))).to(eng.device)
        logits = torch.empty(B, Cn, dtype=torch.float32, device=eng.device)
        last = c.seq_emb.view(B, T, H)[:, T - 1, :]
        self._score_cand(last, T * H, B, cand, Cn, logits)
        self.attention_weights = c.attn
        return [logits.cpu().numpy(), c.attn.cpu().numpy()]

    def score_candidates(self, seq, cand, time_seq=None, hours=None, days=None, timestamps=None, want_attn=False):
        """Batched evaluation scoring: per-user candidate lists cand [U, C] (candidate 0 = target).
        Returns (logits [U,C], count_greater [U], count_equal [U]) as numpy arrays (util.py:317-321 fused);
        want_attn also fills the [h*U, T, T] attention stack of the model's exposed tower (ctx(U).attn)."""
        eng = self.engine
        c = self.forward_eval(seq, time_seq, hours, days, want_attn=want_attn, timestamps=timestamps)
        B, T, H = c.B, eng.T, eng.H
        cand_t = torch.from_numpy(np.ascontiguousarray(np.asarray(cand, dtype=np.int32))).to(eng.device)
        Cn = cand_t.shape[1]
        logits = torch.empty(B, Cn, dtype=torch.float32, device=eng.device)
        cgt = torch.empty(B, dtype=torch.int32, device=eng.device)
        ceq = torch.empty(B, dtype=torch.int32, device=eng.device)
        last = c.seq_emb.view(B, T, H)[:, T - 1, :]
        self._score_cand(last, T * H, B, cand_t, Cn, logits, cgt, ceq)
        return logits.cpu().numpy(), cgt.cpu().numpy(), ceq.cpu().numpy()

    def score_full_catalog(self, seq, target, rated=None, time_seq=None, hours=None, days=None, mode: int = 0):
        """Full-catalog evaluation scoring: rank of target[u] among every item in [1, itemnum] the user has not
        rated (rated: optional list of id collections, one per user).  mode 0 = tcgen05 tensor-core GEMM with exact
        band re-scoring, mode 1 = exact brute force.  Returns (count_greater [U], count_equal [U]) int32 arrays."""
        eng = self.engine
        if eng.item_shard is not None:
            return self._score_full_catalog_sharded(seq, target, rated, time_seq, hours, days, mode)
        c = self.forward_eval(seq, time_seq, hours, days)
        B, T, H = c.B, eng.T, eng.H
        dev = eng.device
        V = eng.P["item_emb"].shape[0]
        tgt = torch.from_numpy(np.ascontiguousarray(np.asarray(target, dtype=np.int32).reshape(-1))).to(dev)
        rptr, ridx = self._id_csr(rated, B) if rated is not None else (None, None)
        cgt = torch.empty(B, dtype=torch.int32, device=dev)
        ceq = torch.empty(B, dtype=torch.int32, device=dev)
        wsb = eng.lib.cast_score_rank_full_workspace_bytes(B, V, H)
        ws = self._pinned.get(("sfws", B))
        if ws is None:
            ws = self._pinned[("sfws", B)] = torch.empty(wsb // 4 + 16, dtype=torch.int32, device=dev)
        last = c.seq_emb.view(B, T, H)[:, T - 1, :]
        eng._call(eng.lib.cast_score_rank_full, last.data_ptr(), T * H, eng.P["item_emb"].data_ptr(), V, H, B,
                  tgt.data_ptr(), None, eng._p(rptr), eng._p(ridx), mode, cgt.data_ptr(), ceq.data_ptr(), None,
                  ws.data_ptr(), wsb, eng._stream())
        if mode == 0:
            import ctypes
            flag = ctypes.c_int(0)
            eng._call(eng.lib.cast_score_rank_full_status, ws.data_ptr(), B, V, ctypes.byref(flag), eng._stream())
            if flag.value != 0:
                raise RuntimeError("score_rank_full: tensor-core pass watchdog fired")
        return cgt.cpu().numpy(), ceq.cpu().numpy()

    def _score_full_catalog_sharded(self, seq, target, rated, time_seq, hours, days, mode):
        """Full-catalog ranks with the item table sharded by row (SURVEY §8e row 3, config 5): every rank runs the
        forward pass for ITS users, the last-position vectors of all ranks are all-gathered, each rank counts — on the
        tensor cores — the items of its own shard that beat the target (whose canonical score is gathered from the
        owning shard), and ONE integer all-reduce adds the per-shard counts up.  Collective: all ranks call it with
        their own users (same count on every rank)."""
        import torch.distributed as dist
        eng = self.engine
        rank, world = eng.item_shard
        dev = eng.device
        c = self.forward_eval(seq, time_seq, hours, days)
        B, T, H = c.B, eng.T, eng.H
        last = c.seq_emb.view(B, T, H)[:, T - 1, :].contiguous()
        tgt_loc = torch.from_numpy(np.ascontiguousarray(np.asarray(target, dtype=np.int32).reshape(-1))).to(dev)
        U = B * world
        last_all = torch.empty(U, H, dtype=torch.float32, device=dev)
        tgt_all = torch.empty(U, dtype=torch.int32, device=dev)
        dist.all_gather_into_tensor(last_all, last)
        dist.all_gather_into_tensor(tgt_all, tgt_loc)
        rated_all = [None] * world
        dist.all_gather_object(rated_all, None if rated is None else [sorted(set(int(i) for i in r)) for r in rated])
        # canonical target scores: one gather from the owning shards
        tscore = torch.empty(U, 1, dtype=torch.float32, device=dev)
        self._score_cand(last_all, H, U, tgt_all.view(U, 1), 1, tscore)
        # this shard's view: local row of the target (0 = not here), local rows of the rated items
        tg = tgt_all.cpu().numpy().astype(np.int64)
        off = 1 if rank else 0
        tl = np.where((tg % world == rank) & (tg > 0) & (tg < eng.V_items), tg // world + off, 0).astype(np.int32)
        rptr = ridx = None
        if rated is not None:
            rptr, ridx = self._id_csr([r for rl in rated_all for r in rl], U, local_rows=True)
        v_loc = (eng.V_items - rank + world - 1) // world + off      # rows of this shard that hold items (+ the pad)
        cgt = torch.zeros(U, dtype=torch.int32, device=dev)
        ceq = torch.zeros(U, dtype=torch.int32, device=dev)
        if v_loc > 1:
            wsb = eng.lib.cast_score_rank_full_workspace_bytes(U, v_loc, H)
            ws = self._pinned.get(("sfws", U))
            if ws is None:
                ws = self._pinned[("sfws", U)] = torch.empty(wsb // 4 + 16, dtype=torch.int32, device=dev)
            eng._call(eng.lib.cast_score_rank_full, last_all.data_ptr(), H, eng.P["item_emb"].data_ptr(), v_loc, H, U,
                      torch.from_numpy(tl).to(dev).data_ptr(), tscore.data_ptr(), eng._p(rptr), eng._p(ridx), mode,
                      cgt.data_ptr(), ceq.data_ptr(), None, ws.data_ptr(), wsb, eng._stream())
            if mode == 0 and dev.type == "cuda":
                import ctypes
                flag = ctypes.c_int(0)
                eng._call(eng.lib.cast_score_rank_full_status, ws.data_ptr(), U, v_loc, ctypes.byref(flag), eng._stream())
                if flag.value != 0:
                    raise RuntimeError("score_rank_full: tensor-core pass watchdog fired")
        both = torch.stack([cgt, ceq])
        dist.all_reduce(both, op=dist.ReduceOp.SUM)
        mine = slice(rank * B, (rank + 1) * B)
        return both[0, mine].cpu().numpy(), both[1, mine].cpu().numpy()

    # parameter access by role name
    def state_dict(self):
        return {k: v.detach().cpu().clone() for k, v in self.engine.P.items()}

    def load_state_dict(self, sd):
        self.engine.load_parameters(sd)


class SASRec(_Model):
    """reference models/sasrec.py:4-129.  `static=True` => sinusoidal positions (registry name `sasrec_static`)."""

    def __init__(self, usernum, itemnum, args, static=False, reuse=None, **kw):
        self.registry_name = "sasrec_static" if static else "sasrec"
        super().__init__(usernum, itemnum, args, **kw)


def _make_cast(n):
    class _CAST(_Model):
        registry_name = f"cast_{n}"

        def __init__(self, usernum, itemnum, ratingnum, args, reuse=None, **kw):
            self.ratingnum = ratingnum
            super().__init__(usernum, itemnum, args, **kw)

    _CAST.__name__ = _CAST.__qualname__ = f"CAST{n}"
    _CAST.__doc__ = f"reference models/cast_{n}.py (see engine.model_plan for the variant's wiring)."
    return _CAST


CAST1, CAST2, CAST3, CAST4, CAST5, CAST6, CAST7, CAST8, CAST9 = (_make_cast(i) for i in range(1, 10))


def build_model(name: str, usernum, itemnum, ratingnum, args, **kw):
    """reference main.py:121-142 dispatch."""
    name = name.lower()
    if name not in MODELS:
        raise ValueError(f"provide model from {MODELS}")
    if name == "sasrec":
        return SASRec(usernum, itemnum, args, **kw)
    if name == "sasrec_static":
        return SASRec(usernum, itemnum, args, static=True, **kw)
    return globals()["CAST" + name.split("_")[1]](usernum, itemnum, ratingnum, args, **kw)
