"""Model classes with the reference's interface (models/sasrec.py:5,127; models/cast_1.py:6,158 ...).

    model = SASRec(usernum, itemnum, args)            # or CAST1..CAST9(usernum, itemnum, ratingnum, args)
    auc, loss = model.train_step(u, seq, pos, neg, time_seq, hours, days)      # == sess.run([auc, loss, train_op])
    logits, attn = model.predict(sess, u, seq, item_idx, timeseq=..., hours_seq=..., days_seq=...)

`args` is the reference's argparse namespace (main.py:42-86); `sess` is accepted and ignored.  Inputs are host
numpy int arrays as produced by the reference's sampler; results are host floats / numpy arrays.
"""
from __future__ import annotations

import ctypes
from typing import Optional

import numpy as np
import torch
import torch.distributed as dist

from .engine import Engine, MODELS


def _all_gather(t):
    """every rank's t, concatenated along dim 0 in rank order"""
    out = torch.empty((dist.get_world_size() * t.shape[0],) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
    dist.all_gather_into_tensor(out, t)
    return out


def _all_gather_lists(lists):
    """every rank's per-user id collections, in rank order (None if this rank passes None)"""
    parts = [None] * dist.get_world_size()
    dist.all_gather_object(parts, None if lists is None else [sorted(set(int(i) for i in r)) for r in lists])
    return None if lists is None else [r for p in parts for r in p]


def check_item_bias(item_bias, itemnum: int) -> torch.Tensor:
    """An item_bias of recommend / similar_items (numpy array or torch tensor of itemnum + 1 reals; entry 0 is ignored)
    rounded once to float32, on the device it came from.  Raises ValueError for a wrong shape, a non-real dtype, or a
    NaN or +inf anywhere after the rounding (-inf removes an item)."""
    if isinstance(item_bias, torch.Tensor):
        t = item_bias
        real = not (t.dtype == torch.bool or t.is_complex())
    else:
        a = np.asarray(item_bias)
        real = a.dtype.kind in "fiu"
        t = torch.from_numpy(np.ascontiguousarray(a)) if real else None
    if not real:
        raise ValueError(f"item_bias must hold real numbers, got dtype {(t if t is not None else a).dtype}")
    if t.dim() != 1 or t.shape[0] != itemnum + 1:
        raise ValueError(f"item_bias must have shape ({itemnum + 1},) (itemnum + 1), got {tuple(t.shape)}")
    t = t.to(torch.float32)
    if bool((torch.isnan(t) | torch.isposinf(t)).any()):
        raise ValueError("item_bias must hold no NaN or +inf (-inf removes an item)")
    return t


class ItemBias:
    """An item_bias validated and laid out for one model's item table: float32 on its device, one entry per row of
    this process's table (b[global id of the row]).  Model.prepare_item_bias makes one; recommend / similar_items
    accept it in place of the array, so a loop of calls validates and copies the bias once."""

    def __init__(self, engine, rows: torch.Tensor):
        self.engine, self.rows = engine, rows


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
        """Capture the whole step (forward, loss, backward, the data-parallel exchange, Adam) as one CUDA graph: one
        host launch per step instead of ~70.  The exchange is plain kernel launches (dist.PeerExchange)."""
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
        g = torch.cuda.CUDAGraph()
        with torch.cuda.stream(s):
            with torch.cuda.graph(g, stream=s):
                eng.launch_train_step(c)
        torch.cuda.current_stream(eng.device).wait_stream(s)
        eng.w.copy_(saved[0]); eng.m.copy_(saved[1]); eng.v.copy_(saved[2]); eng.adam_state.copy_(saved[3])
        c.graph = g

    def launch(self, c):
        """Enqueue one training step on the batch already resident in c.keys3 / c.cids."""
        if self.use_graph:
            if c.graph is None:
                self._capture(c)
            c.graph.replay()
        else:
            self.engine.launch_train_step(c)

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

    def _id_csr(self, lists, n):
        """Per-user id collections -> CSR device tensors (ptr [n+1], idx) of rows of this process's item table, unique
        and ascending per user.  A row-sharded table keeps the ids its shard holds, as local rows (an increasing map,
        so each row stays ascending)."""
        eng = self.engine
        ptr = np.zeros(n + 1, np.int32)
        flat = []
        for u, r in enumerate(lists):
            ids = np.unique(np.asarray(list(r), dtype=np.int64))
            if eng.item_shard is not None:
                ids = eng.local_rows(ids)
                ids = ids[ids > 0]
            flat.append(ids)
            ptr[u + 1] = ptr[u] + len(ids)
        idx = np.concatenate(flat + [np.zeros(1, np.int64)]).astype(np.int32)
        return torch.from_numpy(ptr).to(eng.device), torch.from_numpy(idx).to(eng.device)

    def prepare_item_bias(self, item_bias) -> Optional[ItemBias]:
        """item_bias (see check_item_bias; None -> None) -> ItemBias for this model.  With a row-sharded item table each
        rank keeps b[global ids of its local rows], gathered on the device; every rank passes the same array."""
        if item_bias is None or isinstance(item_bias, ItemBias):
            if item_bias is not None and item_bias.engine is not self.engine:
                raise ValueError("item_bias was prepared for another model")
            return item_bias
        eng = self.engine
        full = check_item_bias(item_bias, self.itemnum).to(eng.device)
        rows = eng.global_ids(torch.arange(eng.item_rows, device=eng.device))
        return ItemBias(eng, full[rows])     # a new contiguous tensor: 16-byte aligned, as the kernels require

    # ------------------------------------------------------------------ full catalog
    # With a row-sharded item table (SURVEY §8e row 3, config 5) score_full_catalog and recommend are collective calls:
    # every rank passes its own users (the same count on every rank), the last-position rows of all ranks are
    # all-gathered, each rank runs the kernel over the items of its own shard and the per-rank results are combined.
    def _last_rows(self, c):
        """(rows, ld) of the last position of each sequence of the batch c; with a row-sharded table, of every rank's
        batch (all-gathered, rank-major)"""
        eng = self.engine
        B, T, H = c.B, eng.T, eng.H
        last = c.seq_emb.view(B, T, H)[:, T - 1, :]
        if eng.item_shard is None:
            return last, T * H
        return _all_gather(last.contiguous()), H

    def _workspace(self, nbytes: int):
        """device workspace of the full-catalog kernels: one buffer, grown on demand (the operand images of a large
        catalog are GBs)"""
        ws = self._pinned.get("catalog_ws")
        if ws is None or ws.numel() * 4 < nbytes:
            self._pinned["catalog_ws"] = None
            ws = self._pinned["catalog_ws"] = torch.empty(nbytes // 4 + 16, dtype=torch.int32, device=self.engine.device)
        return ws

    def _check_watchdog(self, status, what, *args):
        """status(*args, &flag, stream) reads the watchdog flag of a mode-0 call's tensor-core pass; raises if it fired"""
        eng = self.engine
        flag = ctypes.c_int(0)
        eng._call(status, *args, ctypes.byref(flag), eng._stream())
        if flag.value != 0:
            raise RuntimeError(f"{what}: tensor-core pass watchdog fired")

    def score_full_catalog(self, seq, target, rated=None, time_seq=None, hours=None, days=None, mode: int = 0):
        """Full-catalog evaluation scoring: rank of target[u] among every item in [1, itemnum] the user has not
        rated (rated: optional list of id collections, one per user).  mode 0 = tcgen05 tensor-core GEMM with exact
        band re-scoring, mode 1 = exact brute force.  Returns (count_greater [U], count_equal [U]) int32 arrays.
        With a row-sharded item table each rank counts the items of its own shard that beat the target (whose
        canonical score is gathered from the owning shard) and one integer all-reduce adds the counts up."""
        eng = self.engine
        dev = eng.device
        c = self.forward_eval(seq, time_seq, hours, days)
        last, ld = self._last_rows(c)
        U, V = last.shape[0], eng.item_rows
        tgt = torch.from_numpy(np.ascontiguousarray(np.asarray(target, dtype=np.int32).reshape(-1))).to(dev)
        tscore = None
        if eng.item_shard is not None:
            tgt = _all_gather(tgt)
            rated = _all_gather_lists(rated)
            tscore = torch.empty(U, 1, dtype=torch.float32, device=dev)
            self._score_cand(last, ld, U, tgt.view(U, 1), 1, tscore)
            tgt = torch.from_numpy(eng.local_rows(tgt.cpu().numpy().astype(np.int64)).astype(np.int32)).to(dev)
        cgt = torch.zeros(U, dtype=torch.int32, device=dev)
        ceq = torch.zeros(U, dtype=torch.int32, device=dev)
        if V > 1:       # a shard of a catalog smaller than the world may hold no item
            rptr, ridx = self._id_csr(rated, U) if rated is not None else (None, None)
            wsb = eng.lib.cast_score_rank_full_workspace_bytes(U, V, eng.H)
            ws = self._workspace(wsb)
            eng._call(eng.lib.cast_score_rank_full, last.data_ptr(), ld, eng.P["item_emb"].data_ptr(), V, eng.H, U,
                      tgt.data_ptr(), eng._p(tscore), eng._p(rptr), eng._p(ridx), mode, cgt.data_ptr(), ceq.data_ptr(),
                      None, ws.data_ptr(), wsb, eng._stream())
            if mode == 0:
                self._check_watchdog(eng.lib.cast_score_rank_full_status, "score_rank_full", ws.data_ptr(), U, V)
        if eng.item_shard is None:
            return cgt.cpu().numpy(), ceq.cpu().numpy()
        rank = eng.item_shard[0]
        both = torch.stack([cgt, ceq])
        dist.all_reduce(both, op=dist.ReduceOp.SUM)
        mine = slice(rank * c.B, (rank + 1) * c.B)
        return both[0, mine].cpu().numpy(), both[1, mine].cpu().numpy()

    def recommend(self, seq, k=10, exclude=None, time_seq=None, hours=None, days=None, timestamps=None, mode: int = 0,
                  item_bias=None):
        """Exact top-k recommendation from the last position of each sequence: the k items of [1, itemnum] not in
        exclude[u] (optional, one id collection per user) with the largest canonical fp32 logits (the logits of
        score_candidates / predict), ties broken by item id ascending.  mode 0 = tcgen05 tensor cores as an exact
        filter, mode 1 = exact brute force; both return the same bits.  Returns (ids [U,k] int32, scores [U,k] float32);
        fewer than k eligible items pad the tail with id 0 and score -inf.  With a row-sharded item table each rank
        takes the top k of its own shard (local rows -> global ids, an increasing map, so the tie order holds) and the
        ranks' lists are merged per user by (score desc, id asc).
        item_bias (optional, itemnum + 1 reals or an ItemBias): the score of item j becomes fl(logit + b_j), one fp32
        addition, and b_j = -inf removes item j (catalog-wide deny / allow lists, popularity corrections, boosts).  A
        zero bias returns the same ids and equal scores (in IEEE arithmetic fl(-0 + 0) = +0; the canonical logit is never
        -0, so in practice the bits are equal too)."""
        eng = self.engine
        dev = eng.device
        bias = self.prepare_item_bias(item_bias)
        brows = None if bias is None else bias.rows
        c = self.forward_eval(seq, time_seq, hours, days, timestamps=timestamps)
        last, ld = self._last_rows(c)
        U, V = last.shape[0], eng.item_rows
        if eng.item_shard is not None:
            exclude = _all_gather_lists(exclude)
        ids = torch.zeros(U, k, dtype=torch.int32, device=dev)
        scores = torch.full((U, k), float("-inf"), dtype=torch.float32, device=dev)
        if V > 1:       # a shard of a catalog smaller than the world may hold no item
            eptr, eidx = self._id_csr(exclude, U) if exclude is not None else (None, None)
            wsb = eng.lib.cast_topk_full_workspace_bytes(U, V, eng.H, k)
            ws = self._workspace(wsb)
            eng._call(eng.lib.cast_topk_full_biased, last.data_ptr(), ld, eng.P["item_emb"].data_ptr(), V, eng.H, U, k,
                      eng._p(eptr), eng._p(eidx), eng._p(brows), mode, ids.data_ptr(), scores.data_ptr(),
                      None, ws.data_ptr(), wsb, eng._stream())
            if mode == 0:
                self._check_watchdog(eng.lib.cast_topk_full_status, "topk_full", ws.data_ptr(), U, V, eng.H, k)
            ids = eng.global_ids(ids)
        return self._merge_topk(ids, scores, k, c.B)

    def _merge_topk(self, ids, scores, k, n):
        """per-call top-k lists (global ids) -> (ids, scores) numpy arrays of this rank's n rows; with a row-sharded item
        table the rows are every rank's (rank-major) and each rank's per-shard lists are merged per row by (score desc,
        id asc)"""
        eng = self.engine
        if eng.item_shard is None:
            return ids.cpu().numpy(), scores.cpu().numpy()
        rank, world = eng.item_shard
        all_i, all_s = (np.hstack(np.split(_all_gather(t).cpu().numpy(), world)) for t in (ids, scores))
        order = np.lexsort((all_i, -all_s), axis=-1)[:, :k]
        mine = slice(rank * n, (rank + 1) * n)
        return np.take_along_axis(all_i, order, 1)[mine], np.take_along_axis(all_s, order, 1)[mine]

    SIMILARITY = {"dot": 0, "cosine": 1}     # include/cast_b200.h CAST_SIM_*

    def similar_items(self, ids, k=10, metric="cosine", mode: int = 0, item_bias=None):
        """Exact item-to-item top-k: for each query item q of ids, the k items j in [1, itemnum], j != q, with the
        largest canonical score, ties broken by item id ascending (the order of recommend).  metric "dot": the
        canonical fp32 dot of the raw item_emb rows (the training logits' rows, no sqrt(H) factor); "cosine": the
        canonical dot of the rows normalised canonically (n = sqrt_rn of the k-ascending, separately rounded sum of
        squares, each element divided by n, a zero row stays zero).  mode 0 = tcgen05 tensor cores as an exact filter,
        mode 1 = exact brute force; both return the same bits.  Returns (ids [U,k] int32, scores [U,k] float32); fewer
        than k eligible items pad the tail with id 0 and score -inf.  With a row-sharded item table this is a
        collective call (every rank passes its own queries, the same count on every rank): the query rows are read
        from their owners' shards, each rank takes the top k of its own shard for all queries and the lists are merged
        as in recommend.  item_bias as in recommend: the score of j becomes fl(score + b_j), b_j = -inf removes j."""
        eng = self.engine
        dev = eng.device
        if metric not in self.SIMILARITY:
            raise ValueError(f"metric must be one of {sorted(self.SIMILARITY)}, got {metric!r}")
        if not 1 <= int(k) <= 256:
            raise ValueError(f"k must be in [1, 256], got {k}")
        k = int(k)
        q = np.asarray(ids).reshape(-1)
        if q.size and (not np.issubdtype(q.dtype, np.integer) or q.min() < 1 or q.max() > self.itemnum):
            raise ValueError(f"query ids must be integers in [1, {self.itemnum}]")
        bias = self.prepare_item_bias(item_bias)
        brows = None if bias is None else bias.rows
        qd = torch.from_numpy(q.astype(np.int32)).to(dev)
        B = qd.shape[0]
        if eng.item_shard is not None:
            qd = _all_gather(qd)
        U, V = qd.shape[0], eng.item_rows
        nbr = torch.zeros(U, k, dtype=torch.int32, device=dev)
        scores = torch.full((U, k), float("-inf"), dtype=torch.float32, device=dev)
        if U > 0 and V > 1:     # a shard of a catalog smaller than the world may hold no item
            eptr, eidx = self._id_csr(qd.cpu().numpy().reshape(U, 1), U)       # the query itself, if this shard holds it
            metric_id = self.SIMILARITY[metric]
            wsb = eng.lib.cast_similar_items_workspace_bytes(U, V, eng.H, k, metric_id)
            ws = self._workspace(wsb)
            shards = (eng.shard_ptrs.data_ptr(), eng.item_shard[1]) if eng.item_shard is not None else (None, 0)
            eng._call(eng.lib.cast_similar_items_biased, qd.data_ptr(), U, eng.P["item_emb"].data_ptr(), V, *shards,
                      eng.V_items, eng.H, k, metric_id, eptr.data_ptr(), eidx.data_ptr(), eng._p(brows),
                      mode, nbr.data_ptr(), scores.data_ptr(), None, ws.data_ptr(), wsb, eng._stream())
            if mode == 0:
                self._check_watchdog(eng.lib.cast_similar_items_status, "similar_items", ws.data_ptr(), U, V, eng.H, k)
            nbr = eng.global_ids(nbr)
        return self._merge_topk(nbr, scores, k, B)

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

    def last_grad_norm(self):
        """Pre-clip global gradient norm of the most recent training step (waits for it); None when the model was built
        without args.clip_grad."""
        eng = self.engine
        if not eng.clip:
            return None
        return float(eng.clip_out[1].item())

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
