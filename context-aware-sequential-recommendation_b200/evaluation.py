"""Evaluation drivers with the reference's interface and RNG consumption (util.py:230-339 `evaluate`, :342-430
`evaluate_valid`):  `evaluate(model, dataset, args, sess) -> (NDCG@10, HR@10)`.

The reference scores ONE user per `sess.run` (batch 1, ~92 users/s, SURVEY §6).  The candidate construction does not
depend on model outputs, so here it runs first for all users — consuming `random.sample` and `np.random.randint`
exactly as the reference does (same user sub-sample, same 100 negatives per user, negatives may repeat and may equal
the target) — and the model then scores the users in large batches on the GPU: one forward pass + the fused
101-candidate dot / count-greater kernel (`cast_score_rank_cand`).

Rank rule (SURVEY A-12): the device returns, per user, `count_greater` and `count_equal` (other candidates whose
logit is exactly the target's).  Without ties `count_greater` IS `(-p).argsort().argsort()[0]`; users with ties are
resolved on the host with the literal reference expression on the device logits, so ranks match the reference's
expression bit for bit on identical logits.  HR / NDCG accumulate in user order in float64 as the reference does.

Under `torch.distributed` (`world_size > 1`) users are sharded contiguously over ranks; the only exchange is one
integer all-reduce of the rank histogram (dist.reduce_rank_histogram), so HR@10 is exact and NDCG@10 is a float64
function of integers.
"""
from __future__ import annotations

import copy
import random
from typing import Optional

import numpy as np

from .data import get_delta_range, raw_ts, timedelta_bins


def _user_pool(usernum: int):
    """util.py:241-244 / :350-353 — sub-sample 10000 users of large datasets with Python's `random`."""
    if usernum > 10000:
        return random.sample(range(1, usernum + 1), 10000)
    return range(1, usernum + 1)


def _draw_negatives(rng, itemnum: int, member: np.ndarray, n: int = 100) -> np.ndarray:
    """util.py:291-298 — n accepted draws of randint(1, itemnum+1) (rejected: the user's train items), in stream
    order.  Block draws equal scalar draws for numpy's legacy generator (see sampler.py)."""
    out = np.empty(n, dtype=np.int32)
    got = 0
    while got < n:
        d = rng.randint(1, itemnum + 1, size=n - got)
        ok = d[~member[d]]
        out[got:got + len(ok)] = ok
        got += len(ok)
    return out


def _featurise(hist, T: int, args, log_scale: bool, lo, hi):
    """One left-padded input row of the newest len(hist) <= T events: item ids, time bins relative to the newest input
    event (util.py:276-289), hours, weekdays, raw timestamps."""
    k = len(hist)
    seq = np.zeros(T, np.int32)
    timeseq = np.zeros(T, np.int32)
    hours = np.zeros(T, np.int32)
    days = np.zeros(T, np.int32)
    seq[T - k:] = [x.item for x in hist]
    hours[T - k:] = [x.ts.hour for x in hist]
    days[T - k:] = [x.ts.day for x in hist]
    t = np.fromiter((raw_ts(x) for x in hist), dtype=np.int64, count=k)
    # bins relative to the newest INPUT event; the valid->test delta the reference computes first is overwritten
    timeseq[T - k:] = timedelta_bins((t[-1] - t).astype(np.float64), args.bin_in_hours, args.max_bins, log_scale, lo, hi)
    tsraw = np.zeros(T, np.int64)
    tsraw[T - k:] = t
    return seq, timeseq, hours, days, tsraw


def build_candidates(dataset, args, split: str = "test", rng=None):
    """Everything `model.predict` is fed for every evaluated user, in the reference's user order.

    split = "test": input = train + valid item, target = test item (util.py:246-298);
    split = "valid": input = train, target = valid item (util.py:356-398).
    Returns dict(u [U], seq [U,T], item_idx [U,101], timeseq, hours, days [U,T]) of int32 arrays."""
    train, valid, test, usernum, itemnum = dataset[0], dataset[1], dataset[2], dataset[3], dataset[4]
    rng = np.random if rng is None else rng
    T = args.maxlen
    log_scale = bool(args.log_scale)
    lo, hi = get_delta_range(train)
    target_of = test if split == "test" else valid
    member = np.zeros(itemnum + 2, dtype=bool)
    us, seqs, cands, tss, hrs, dys, rated, raws = [], [], [], [], [], [], [], []
    trunc = None
    if getattr(args, "test_model", None):
        if not getattr(args, "test_seq_len", None):
            raise Exception("test_seq_len is not provided")
        trunc = min(int(args.test_seq_len), T)
    for u in _user_pool(usernum):
        tr = train[u]
        if len(tr) < 1 or len(target_of[u]) < 1:
            continue
        hist = list(tr[-T:]) if split == "valid" else list(tr[-(T - 1):] if T > 1 else []) + [valid[u][0]]
        seq, timeseq, hours, days, tsraw = _featurise(hist, T, args, log_scale, lo, hi)
        items = np.fromiter((x.item for x in tr), dtype=np.int64, count=len(tr))
        member[items] = True
        member[0] = True
        neg = _draw_negatives(rng, itemnum, member)
        member[items] = False
        if trunc is not None:  # util.py:300-315 (--test_model / --test_seq_len)
            seq[:-trunc] = 0
            timeseq[:-trunc] = 0
            hours[:-trunc] = 0
            days[:-trunc] = 0
            tsraw[:-trunc] = 0
        us.append(u)
        rated.append(np.unique(items).astype(np.int32))
        seqs.append(seq)
        cands.append(np.concatenate([[target_of[u][0].item], neg]).astype(np.int32))
        tss.append(timeseq)
        hrs.append(hours)
        dys.append(days)
        raws.append(tsraw)
    st = lambda a, w: np.stack(a) if a else np.zeros((0, w), np.int32)  # noqa: E731
    return {"u": np.asarray(us, np.int32), "seq": st(seqs, T), "item_idx": st(cands, 101), "timeseq": st(tss, T),
            "hours": st(hrs, T), "days": st(dys, T), "rated": rated,
            "tsraw": np.stack(raws) if raws else np.zeros((0, T), np.int64)}   # for the device-side feature path


def build_recommend_inputs(dataset, args):
    """Inputs for recommending each user's next items: the last maxlen events of train + valid + test (users without
    events are skipped), featurised as in build_candidates (no --test_seq_len truncation), and the ids of the whole
    history as the exclusion set.  Draws no random numbers.
    Returns dict(u [U], seq, timeseq, hours, days [U,T] int32, tsraw [U,T] int64, rated: list of id arrays)."""
    train, valid, test, usernum = dataset[0], dataset[1], dataset[2], dataset[3]
    T = args.maxlen
    log_scale = bool(args.log_scale)
    lo, hi = get_delta_range(train)
    us, seqs, tss, hrs, dys, raws, rated = [], [], [], [], [], [], []
    for u in range(1, usernum + 1):
        full = list(train.get(u, [])) + list(valid.get(u, [])) + list(test.get(u, []))
        if not full:
            continue
        seq, timeseq, hours, days, tsraw = _featurise(full[-T:], T, args, log_scale, lo, hi)
        us.append(u)
        seqs.append(seq)
        tss.append(timeseq)
        hrs.append(hours)
        dys.append(days)
        raws.append(tsraw)
        rated.append(np.unique(np.fromiter((x.item for x in full), dtype=np.int64, count=len(full))).astype(np.int32))
    st = lambda a, dt: np.stack(a) if a else np.zeros((0, T), dt)  # noqa: E731
    return {"u": np.asarray(us, np.int32), "seq": st(seqs, np.int32), "timeseq": st(tss, np.int32),
            "hours": st(hrs, np.int32), "days": st(dys, np.int32), "tsraw": st(raws, np.int64), "rated": rated}


def _batches(model, rows, batch_users: int, lo: int, hi: int):
    """Fixed-shape batches over rows [lo, hi) of a build_candidates / build_recommend_inputs dict; the tail batch is
    padded with zero rows and empty id lists.  Yields (out, pad, feats): the batch's slice of the [hi - lo] results,
    pad(key) -> the batch of rows[key], and the time-feature keywords of the model call — the raw timestamps
    (featurised on the device, util.py:276-289) when the model has use_device_time_features and the rows carry them,
    else the time-bin / hour / weekday id sequences."""
    B = max(1, min(batch_users, max(1, hi - lo)))
    use_ts = getattr(model, "timefeat", None) is not None and "tsraw" in rows
    for s in range(lo, hi, B):
        e = min(hi, s + B)
        n = e - s

        def pad(key):
            a = rows[key]
            if key == "rated":     # one id collection per user
                return list(a[s:e]) + [np.zeros(0, np.int32)] * (B - n)
            if n == B:
                return a[s:e]
            out = np.zeros((B,) + a.shape[1:], a.dtype)
            out[:n] = a[s:e]
            return out

        feats = ({"timestamps": pad("tsraw")} if use_ts else
                 {"time_seq": pad("timeseq"), "hours": pad("hours"), "days": pad("days")})
        yield slice(s - lo, e - lo), pad, feats


def recommend_users(model, inputs, k: int, batch_users: int = 256, lo: int = 0, hi: Optional[int] = None,
                    mode: int = 0, item_bias=None):
    """model.recommend over rows [lo, hi) of build_recommend_inputs' output, with each user's history excluded; fixed
    batch shape (tail padded as in score_users); item_bias as in model.recommend, validated and moved to the device
    once for all batches.  Returns (ids [n,k] int32, scores [n,k] float32)."""
    hi = len(inputs["u"]) if hi is None else hi
    bias = model.prepare_item_bias(item_bias)
    ids = np.zeros((max(0, hi - lo), k), np.int32)
    scores = np.zeros((max(0, hi - lo), k), np.float32)
    for out, pad, feats in _batches(model, inputs, batch_users, lo, hi):
        n = out.stop - out.start
        i, sc = model.recommend(pad("seq"), k, pad("rated"), mode=mode, item_bias=bias, **feats)
        ids[out] = i[:n]
        scores[out] = sc[:n]
    return ids, scores


def similar_items_all(model, k: int, batch: int = 4096, lo: int = 0, hi: Optional[int] = None,
                      metric: str = "cosine", mode: int = 0, item_bias=None):
    """model.similar_items for the query items lo+1 .. hi (rows [lo, hi) of the ids 1..itemnum; hi defaults to
    itemnum) in fixed-shape batches, the tail batch padded with item 1 (its results are dropped); item_bias as in
    model.similar_items, validated and moved to the device once for all batches.
    Returns (items [n] int32, neighbours [n,k] int32, scores [n,k] float32)."""
    hi = model.itemnum if hi is None else hi
    bias = model.prepare_item_bias(item_bias)
    items = np.arange(lo + 1, hi + 1, dtype=np.int32)
    n = len(items)
    nbr = np.zeros((n, k), np.int32)
    scores = np.zeros((n, k), np.float32)
    B = max(1, min(batch, n))
    for s in range(0, n, B):
        e = min(n, s + B)
        q = np.ones(B, np.int32)
        q[:e - s] = items[s:e]
        i, sc = model.similar_items(q, k, metric, mode=mode, item_bias=bias)
        nbr[s:e] = i[:e - s]
        scores[s:e] = sc[:e - s]
    return items, nbr, scores


def reference_rank(logits_row: np.ndarray) -> int:
    """util.py:318-321 verbatim semantics: rank of candidate 0 under numpy's default argsort."""
    return int((-logits_row).argsort().argsort()[0])


def ranks_from_device(logits: np.ndarray, cgt: np.ndarray, ceq: np.ndarray) -> np.ndarray:
    ranks = cgt.astype(np.int64).copy()
    for i in np.flatnonzero(ceq):
        ranks[i] = reference_rank(logits[i])
    return ranks


def metrics_from_ranks(ranks) -> tuple:
    """util.py:323-339 — float64 accumulation in user order."""
    ndcg = 0.0
    ht = 0.0
    n = 0.0
    for r in ranks:
        n += 1
        if r < 10:
            ndcg += 1 / np.log2(r + 2)
            ht += 1
    if n == 0:
        raise ZeroDivisionError("no valid users")
    return ndcg / n, ht / n


def metrics_from_histogram(hist) -> tuple:
    """hist[0..9] = users with rank r, hist[10] = valid users (integers; the multi-GPU reduction)."""
    n = float(hist[10])
    ndcg = sum(float(hist[r]) * float(1 / np.log2(r + 2)) for r in range(10))
    ht = float(sum(int(hist[r]) for r in range(10)))
    return ndcg / n, ht / n


def score_users(model, cand, batch_users: int = 256, lo: int = 0, hi: Optional[int] = None, mode: str = "101",
                attn_sum=None):
    """Ranks of cand rows [lo, hi) through the model's batched scoring path; fixed batch shape (tail padded).
    mode "101": the reference's target + 100 sampled negatives; mode "full": rank among every item the user has not
    rated (count of strictly greater logits; exact ties do not push the target down)."""
    """attn_sum (optional float64 device tensor [T,T]): accumulates the first-head attention map of every scored
    user — what the reference collects per user in --test_model mode (util.py:329-336)."""
    hi = len(cand["u"]) if hi is None else hi
    ranks = np.zeros(max(0, hi - lo), np.int64)
    for out, pad, feats in _batches(model, cand, batch_users, lo, hi):
        n = out.stop - out.start
        seq = pad("seq")
        if mode == "full":      # score_full_catalog takes the id sequences
            cgt, _ = model.score_full_catalog(seq, pad("item_idx")[:, 0], pad("rated"), pad("timeseq"), pad("hours"),
                                              pad("days"))
            ranks[out] = cgt[:n]
            continue
        want = attn_sum is not None
        logits, cgt, ceq = model.score_candidates(seq, pad("item_idx"), want_attn=want, **feats)
        if want:   # head 0 of user b is row b of the [h*B, T, T] stack (modules.py:208-213)
            attn_sum += model.engine.ctx(len(seq)).attn[:n].sum(0, dtype=attn_sum.dtype)
        ranks[out] = ranks_from_device(logits[:n], cgt[:n], ceq[:n])
    return ranks


def _evaluate(model, dataset, args, split, batch_users, rng, mode="101", avg_attention=False):
    cand = build_candidates(dataset, args, split, rng)
    U = len(cand["u"])
    if avg_attention:
        return _evaluate_with_attention(model, cand, batch_users, mode)
    try:
        import torch.distributed as dist
        world = dist.get_world_size() if dist.is_initialized() else 1
    except Exception:  # pragma: no cover
        world = 1
    if world == 1:
        return metrics_from_ranks(score_users(model, cand, batch_users, mode=mode))
    import torch
    from . import dist as cdist
    rank = dist.get_rank()
    lo, hi = cdist.shard_users(U, rank, world)
    ranks = score_users(model, cand, batch_users, lo, hi, mode=mode)
    hist = np.zeros(11, np.int64)
    for r in ranks:
        if r < 10:
            hist[r] += 1
    hist[10] = len(ranks)
    dev = model.engine.device if dist.get_backend() == "nccl" else "cpu"
    h = torch.from_numpy(hist).to(dev)
    cdist.reduce_rank_histogram(h)
    return metrics_from_histogram(h.cpu().numpy())


def _evaluate_with_attention(model, cand, batch_users, mode):
    """metrics + the attention map averaged over the evaluated users (reference util.py:329-336; the reference renders
    it to attention_weights.svg, here the [T,T] array is returned — plotting is out of scope)."""
    import torch
    eng = model.engine
    U = len(cand["u"])
    acc = torch.zeros(eng.T, eng.T, dtype=torch.float64, device=eng.device)
    world, rank = 1, 0
    try:
        import torch.distributed as dist
        if dist.is_initialized():
            world, rank = dist.get_world_size(), dist.get_rank()
    except Exception:  # pragma: no cover
        pass
    if world == 1:
        ranks = score_users(model, cand, batch_users, mode="101", attn_sum=acc)
        return metrics_from_ranks(ranks), (acc / max(1, U)).cpu().numpy()
    from . import dist as cdist
    lo, hi = cdist.shard_users(U, rank, world)
    ranks = score_users(model, cand, batch_users, lo, hi, mode="101", attn_sum=acc)
    hist = np.zeros(11, np.int64)
    for r in ranks:
        if r < 10:
            hist[r] += 1
    hist[10] = len(ranks)
    on_dev = dist.get_backend() == "nccl"
    h = torch.from_numpy(hist).to(eng.device if on_dev else "cpu")
    cdist.reduce_rank_histogram(h)
    a = acc if on_dev else acc.cpu()
    dist.all_reduce(a, op=dist.ReduceOp.SUM)
    return metrics_from_histogram(h.cpu().numpy()), (a / max(1, U)).cpu().numpy()


def evaluate(model, dataset, args, sess=None, batch_users: int = 256, rng=None, mode: str = "101",
             avg_attention: bool = False):
    """Drop-in for reference util.evaluate (test split).  mode="full" ranks against the whole catalog instead of the
    reference's 100 sampled negatives (the negatives are still drawn, so the RNG streams stay aligned).
    avg_attention=True (the reference's --test_model behaviour, util.py:329-336): returns ((NDCG, HR), avg_attn [T,T])."""
    return _evaluate(model, dataset, args, "test", batch_users, rng, mode, avg_attention)


def evaluate_valid(model, dataset, args, sess=None, batch_users: int = 256, rng=None, mode: str = "101"):
    """Drop-in for reference util.evaluate_valid."""
    return _evaluate(model, dataset, args, "valid", batch_users, rng, mode)
