"""Data-parallel path with world_size 2 on CPU (`gloo`), kernels host-emulated (tests/emu, test infrastructure):
two ranks with B/2 sequences each must reproduce the single-process step on B sequences — the reference's loss is
sum(terms)/sum(istarget) over the WHOLE batch (models/sasrec.py:105-108), so ranks exchange un-normalised numerators
plus the target count, summed in rank order over peer memory (dist.py) — and the evaluation histogram reduction must
be exact."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from helpers import backend, golden_batch, make_args, rel_err
from cast_b200.engine import Engine


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _load_batch(eng, gb, lo, hi):
    c = eng.ctx(hi - lo)
    c.keys3.copy_(torch.from_numpy(np.stack([gb[k][lo:hi].reshape(-1) for k in ("seq", "pos", "neg")])))
    c.cids.copy_(torch.from_numpy(np.stack([gb[k][lo:hi].reshape(-1) for k in ("timeseq", "hours", "days")])))
    return c


def _worker(rank, world, port, model, out, shard=False):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    from cast_b200 import dist as cdist
    from cast_b200 import evaluation as cev
    cdist.init_from_env("gloo")
    lib, dev = backend("emu")
    B, T, H = 4, 10, 12
    args = make_args(hidden_units=H, maxlen=T, num_heads=2, num_blocks=1, dropout_rate=0.0)
    gb = golden_batch(B=B, T=T)
    arena = cdist.PeerArena(lib, dev) if shard else None        # CPU stand-in for NVLink peer memory: POSIX shm
    eng = Engine(model, 80, 300, args, device=dev, lib=lib,
                 seed=5 if shard else 5 + rank,                  # replicated: different init per rank on purpose
                 item_shard=(rank, world) if shard else None, alloc=arena.alloc if shard else None)
    cdist.attach(eng, arena=arena)                               # rank 0's dense parameters win
    per = B // world
    c = _load_batch(eng, gb, rank * per, (rank + 1) * per)
    eng.launch_train_step(c)
    hist = torch.tensor([rank + 1] * 10 + [7], dtype=torch.int64)
    cdist.reduce_rank_histogram(hist)
    lo, hi = cdist.shard_users(11, rank, world)
    # every rank's flat buffers (a row-sharded table: shard first, then the replicated dense weights)
    w = [torch.zeros_like(eng.w) for _ in range(world)]
    g = [torch.zeros_like(eng.gbuf) for _ in range(world)]
    dist.all_gather(w, eng.w.clone())
    dist.all_gather(g, eng.adam_g.clone())          # the exchanged gradients (what Adam consumed)
    region = eng.P["item_emb"].numel() if shard else 0
    assert torch.equal(w[0][region:], w[1][region:])     # replicas identical after the step
    if rank == 0:
        single = Engine(model, 80, 300, args, device=dev, lib=lib, seed=5)
        cs = _load_batch(single, gb, 0, B)
        single.launch_train_step(cs)
        res = {"g_dp": eng.adam_g.numpy().copy(), "g_1": single.gbuf.numpy().copy(), "w_dp": eng.w.numpy().copy(),
               "w_1": single.w.numpy().copy(), "hist": hist.numpy().copy(), "shard": (lo, hi),
               "offsets": dict(single.offsets), "sizes": {k: v.numel() for k, v in single.P.items()},
               "w_all": [x.numpy().copy() for x in w], "g_all": [x.numpy().copy() for x in g],
               "region": region, "shard_R": eng.shard_R}
        torch.save(res, out)
    dist.barrier()
    if shard:
        arena.close()
    dist.destroy_process_group()


@pytest.mark.emu
@pytest.mark.parametrize("model", ["sasrec", "cast_1"])
def test_two_rank_step_equals_single_process(tmp_path, model):
    """rank-ordered sum over peer memory behind a flag barrier (dist.PeerExchange; shared memory stands in for
    NVLink)"""
    out = str(tmp_path / "res.pt")
    mp.spawn(_worker, args=(2, _free_port(), model, out, False), nprocs=2, join=True)
    r = torch.load(out, weights_only=False)
    g_dp, g_1 = r["g_dp"], r["g_1"]
    assert abs(g_dp[-2] - g_1[-2]) == 0            # sum(istarget): exact
    assert abs(g_dp[-4] - g_1[-4]) <= 1e-5 * abs(g_1[-4])   # loss numerator
    for k, off in r["offsets"].items():
        n = r["sizes"][k]
        if k.endswith("k.b"):
            continue
        assert rel_err(g_dp[off:off + n], g_1[off:off + n]) <= 2e-5, k
    assert np.array_equal(r["hist"], np.array([3] * 10 + [14]))
    assert r["shard"] == (0, 6)


def _unshard(flat_per_rank, R, H, V):
    """full [V, H] table from the ranks' shards (cyclic ownership, local row 0 of ranks > 0 is a pad)"""
    world = len(flat_per_rank)
    full = np.zeros((V, H), np.float32)
    for q, flat in enumerate(flat_per_rank):
        sh = flat[:R * H].reshape(R, H)
        ids = np.arange(q, V, world)
        full[ids] = sh[(1 if q else 0):(1 if q else 0) + len(ids)]
    return full


@pytest.mark.emu
def test_row_sharded_item_table_step_equals_single_process(tmp_path):
    """dist.attach_sharded (BASELINE config 5 path) on 2 ranks: each rank holds HALF of the item table (+ its gradient
    and Adam slots); lookups read the owning rank's shard (POSIX shared memory standing in for NVLink peer memory);
    after the exchange of the dense gradients each owner folds both ranks' sorted entries into its gradient shard
    in rank order and runs Adam on [own shard | dense weights].  No table collective.  Gradient and parameters of every
    table row must equal the single-process step on the whole batch."""
    out = str(tmp_path / "res.pt")
    mp.spawn(_worker, args=(2, _free_port(), "sasrec", out, True), nprocs=2, join=True)
    r = torch.load(out, weights_only=False)
    H, V, R, region = 12, 301, r["shard_R"], r["region"]
    assert region == R * H and R == 152                     # ceil(301 / 2) + 1: half the table per rank
    n1 = r["sizes"]["item_emb"]
    w_1, g_1 = r["w_1"], r["g_1"]
    g_tab = _unshard(r["g_all"], R, H, V)
    w_tab = _unshard(r["w_all"], R, H, V)
    g1_tab, w1_tab = g_1[:n1].reshape(V, H), w_1[:n1].reshape(V, H)
    cnt = g_1[-2]
    assert r["g_all"][0][-2] == cnt                         # global sum(istarget) on every rank
    assert rel_err(g_tab, g1_tab) <= 2e-5                   # embedding gradient: owner pull == local scatter
    assert not g_tab[~np.any(g1_tab != 0, axis=1)].any()    # untouched rows: exactly zero (integer work is exact)
    sig = np.abs(g1_tab / cnt) > 1e-5
    assert sig.sum() > 500
    assert np.abs(w_tab[sig] - w1_tab[sig]).max() <= 2e-6
    assert np.array_equal(w_tab[g1_tab == 0], w1_tab[g1_tab == 0])
    # dense weights: gradient and parameters as in the replicated test
    for k, off in r["offsets"].items():
        if k == "item_emb" or k.endswith("k.b"):
            continue
        n = r["sizes"][k]
        a = r["g_dp"][region + off - n1: region + off - n1 + n]
        assert rel_err(a, g_1[off:off + n]) <= 2e-5, k
    for q in (1,):                                          # the pad row of ranks > 0 never moves
        assert not r["w_all"][q][:H].any() and not r["g_all"][q][:H].any()


def _eval_worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    import random
    import cast_b200
    from cast_b200 import data as cdata
    from cast_b200 import dist as cdist
    from cast_b200 import evaluation as cev
    cdist.init_from_env("gloo")
    lib, dev = backend("emu")
    here = os.path.dirname(os.path.abspath(__file__))
    dataset = cdata.data_partition(os.path.join(here, "golden", "ref_dataset.txt"), False)
    args = make_args(hidden_units=12, maxlen=8, num_heads=1, num_blocks=1, dropout_rate=0.0)
    args.test_model = None
    args.test_seq_len = None
    m = cast_b200.SASRec(dataset[3], dataset[4], args, device=dev, _lib=lib, use_graph=False, seed=3)
    random.seed(5)
    np.random.seed(5)
    sharded = cev.evaluate(m, dataset, args, None, batch_users=16)       # users sharded over the 2 ranks
    if rank == 0:
        dist.barrier()
        torch.save({"sharded": sharded}, out)
    else:
        dist.barrier()
    dist.destroy_process_group()


@pytest.mark.emu
def test_user_sharded_evaluation_equals_single_process(tmp_path):
    """evaluation.evaluate under world_size 2: users split contiguously, integer histogram all-reduce; HR@10 must be
    identical to the single-process value and NDCG@10 equal up to float64 summation order."""
    import random
    import cast_b200
    from cast_b200 import data as cdata
    from cast_b200 import evaluation as cev
    out = str(tmp_path / "ev.pt")
    mp.spawn(_eval_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    r = torch.load(out, weights_only=False)
    lib, dev = backend("emu")
    here = os.path.dirname(os.path.abspath(__file__))
    dataset = cdata.data_partition(os.path.join(here, "golden", "ref_dataset.txt"), False)
    args = make_args(hidden_units=12, maxlen=8, num_heads=1, num_blocks=1, dropout_rate=0.0)
    args.test_model = None
    args.test_seq_len = None
    m = cast_b200.SASRec(dataset[3], dataset[4], args, device=dev, _lib=lib, use_graph=False, seed=3)
    random.seed(5)
    np.random.seed(5)
    ndcg, hr = cev.evaluate(m, dataset, args, None, batch_users=16)
    assert r["sharded"][1] == hr
    assert abs(r["sharded"][0] - ndcg) < 1e-12


def _sharded_eval_worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    import cast_b200
    from cast_b200 import dist as cdist
    cdist.init_from_env("gloo")
    lib, dev = backend("emu")
    U, T, H, V = 8, 10, 12, 300
    args = make_args(hidden_units=H, maxlen=T, num_heads=1, num_blocks=1, dropout_rate=0.0)
    gb = golden_batch(B=U, T=T)
    rng = np.random.RandomState(3)
    cand = np.concatenate([gb["pos"][:, -1:], rng.randint(1, V + 1, (U, 100))], 1).astype(np.int32)
    cand[0, 4] = cand[0, 0]                                   # a tie with the target
    target = cand[:, 0].copy()
    rated = [set(int(i) for i in gb["seq"][u] if i > 0) for u in range(U)]
    arena = cdist.PeerArena(lib, dev)
    m = cast_b200.SASRec(80, V, args, device=dev, _lib=lib, use_graph=False, seed=3, item_shard=(rank, world),
                         alloc=arena.alloc)
    cdist.attach(m.engine, arena=arena)
    per = U // world
    sl = slice(rank * per, (rank + 1) * per)
    lg, cgt, ceq = m.score_candidates(gb["seq"][sl], cand[sl])
    fgt, feq = m.score_full_catalog(gb["seq"][sl], target[sl], rated[sl.start:sl.stop], mode=1)
    parts = [None] * world
    dist.all_gather_object(parts, (lg, cgt, ceq, fgt, feq))
    if rank == 0:
        single = cast_b200.SASRec(80, V, args, device=dev, _lib=lib, use_graph=False, seed=3)
        lg1, cgt1, ceq1 = single.score_candidates(gb["seq"], cand)
        fgt1, feq1 = single.score_full_catalog(gb["seq"], target, rated, mode=1)
        torch.save({"sharded": [np.concatenate([p[i] for p in parts]) for i in range(5)],
                    "single": [lg1, cgt1, ceq1, fgt1, feq1]}, out)
    dist.barrier()
    arena.close()
    dist.destroy_process_group()


@pytest.mark.emu
def test_item_sharded_evaluation_equals_single_process(tmp_path):
    """Evaluation with the item table row-sharded over 2 ranks (SURVEY §8e row 3): 101-candidate logits gathered from
    the owning shards are bit-identical to the unsharded ones, and the full-catalog rank counts — per-shard
    count_greater / count_equal partials + one integer all-reduce — are exactly the single-process integers."""
    out = str(tmp_path / "res.pt")
    mp.spawn(_sharded_eval_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    r = torch.load(out, weights_only=False)
    sh, s1 = r["sharded"], r["single"]
    assert np.array_equal(sh[0].view(np.uint32), s1[0].view(np.uint32))     # logits: same canonical dot, same rows
    for i in (1, 2, 3, 4):
        assert np.array_equal(sh[i], s1[i]), i
    assert s1[2][0] >= 1 and s1[3].max() > 0
