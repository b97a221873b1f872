"""Exact item-to-item top-K (`cast_item_rows`, `cast_similar_items`, `Model.similar_items`): neighbour ids and score
bits against a numpy float32 restatement of the contract (`normalise` + `similar_reference` below: canonical row
normalisation, canonical dot, score descending, id ascending, the query itself and row 0 never returned, (0, -inf)
padding).  The tensor-core filter (mode 0) must return the same bits as brute force (mode 1) on every case: exact ties
at the K-th place, zero rows, parallel rows of different norms, a tied block larger than the candidate buffer."""
import ctypes
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from helpers import O, backend, make_args, synth_batch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DATASET = os.path.join(ROOT, "tests", "golden", "ref_dataset.txt")
ERR_BAD_ARG, ERR_WORKSPACE = -1, -3
DOT, COSINE = 0, 1
METRIC = {"dot": DOT, "cosine": COSINE}


def normalise(table):
    """n = sqrt_rn(sum_k e_k * e_k) (k ascending, product and sum each rounded to fp32), e_k / n, n == 0 -> 0"""
    e = np.asarray(table, np.float32)
    n2 = np.zeros(e.shape[0], np.float32)
    for k in range(e.shape[1]):
        n2 = (n2 + (e[:, k] * e[:, k]).astype(np.float32)).astype(np.float32)
    n = np.sqrt(n2).astype(np.float32)
    out = np.zeros_like(e)
    nz = n != 0
    out[nz] = (e[nz] / n[nz, None]).astype(np.float32)
    return out


def similar_scores(table, qids, metric):
    rows = normalise(table) if metric == "cosine" else np.asarray(table, np.float32)
    return O.canonical_logits(rows[np.asarray(qids)], rows)


def similar_reference(table, qids, K, metric, scores=None):
    """per query q: the K rows j in [1, V), j != q, by canonical score descending then id ascending; (0, -inf) pads"""
    s = similar_scores(table, qids, metric) if scores is None else scores
    U, V = s.shape
    ids = np.zeros((U, K), np.int32)
    sc = np.full((U, K), -np.inf, np.float32)
    for u, q in enumerate(qids):
        j = np.setdiff1d(np.arange(1, V), [q])
        o = j[np.lexsort((j, -s[u, j]))][:K]
        ids[u, :len(o)] = o
        sc[u, :len(o)] = s[u, o]
    return ids, sc


def assert_same(ids, sc, ids_o, sc_o, what=""):
    bad = np.flatnonzero((ids != ids_o).any(1) | (sc.view(np.uint32) != sc_o.view(np.uint32)).any(1))
    assert bad.size == 0, (what, bad[:8], ids[bad[:1]], ids_o[bad[:1]], sc[bad[:1]], sc_o[bad[:1]])


def sim_call(kind, table, qids, K, metric, mode=0, ws_bytes=None):
    """cast_similar_items on a replicated table, each query's own row excluded; returns (rc, ids, scores, stats, flag)"""
    lib, dev = backend(kind)
    V, H = table.shape
    U = len(qids)
    m = METRIC.get(metric, metric)
    tt = torch.from_numpy(np.ascontiguousarray(table, np.float32)).to(dev)
    q = torch.from_numpy(np.asarray(qids, np.int32)).to(dev)
    ep = torch.arange(U + 1, dtype=torch.int32).to(dev)
    ids = torch.full((U, max(K, 1)), -7, dtype=torch.int32, device=dev)
    sc = torch.full((U, max(K, 1)), 7.0, dtype=torch.float32, device=dev)
    stats = torch.zeros(2, dtype=torch.int64, device=dev)
    need = lib.cast_similar_items_workspace_bytes(U, V, H, K, m)
    wsb = need if ws_bytes is None else ws_bytes
    ws = torch.empty(max(need, wsb) // 4 + 16, dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream if dev.type == "cuda" else None
    rc = lib.cast_similar_items(q.data_ptr(), U, tt.data_ptr(), V, None, 0, V, H, K, m, ep.data_ptr(), q.data_ptr(),
                                mode, ids.data_ptr(), sc.data_ptr(), stats.data_ptr(), ws.data_ptr(), wsb, stream)
    flag = ctypes.c_int(-1)
    if rc == 0:
        assert lib.cast_similar_items_status(ws.data_ptr(), U, V, H, K, ctypes.byref(flag), stream) == 0
    return rc, ids.cpu().numpy(), sc.cpu().numpy(), stats.cpu().numpy(), flag.value


def make_table(V, H, seed, ties_for=(), K=10, zero_rows=0, parallel=0):
    """random table; for each query in ties_for, three more copies of the row at its K-th place (cosine and dot), some
    all-zero rows and some rows that are positive multiples of another row (equal directions, different norms)"""
    rng = np.random.RandomState(seed)
    table = (rng.randn(V, H) * 0.3).astype(np.float32)
    if zero_rows:
        table[rng.choice(np.arange(1, V), zero_rows, replace=False)] = 0.0
    if parallel:
        src = rng.randint(1, V, parallel)
        dst = rng.choice(np.arange(1, V), parallel, replace=False)
        scale = rng.choice(np.float32([0.25, 0.5, 3.0, 7.0, 1.0009765625]), parallel)
        table[dst] = table[src] * scale[:, None]
    for q in ties_for:
        approx = (table[q].astype(np.float64) @ table.T.astype(np.float64)) / (
            np.linalg.norm(table, axis=1).astype(np.float64) + 1e-30)
        approx[[0, q]] = -np.inf
        b = int(np.argsort(-approx)[min(K, V - 3) - 1])
        others = np.setdiff1d(np.arange(1, V), [b, q])
        table[rng.choice(others, 3, replace=False)] = table[b]
    return table


# ------------------------------------------------------------------------------------------------ host emulation
@pytest.mark.emu
@pytest.mark.parametrize("metric", ["cosine", "dot"])
def test_exact_path_emulated_ties_zero_rows_padding(metric):
    V, H = 90, 12
    qids = [1, 5, 17, 33, 89, 40]
    table = make_table(V, H, 3, ties_for=qids[:3], K=7, zero_rows=6, parallel=5)
    table[0] = table[5] * 4.0                           # row 0 would win for query 5: it must never be returned
    table[40] = 0.0                                     # a zero query: every cosine score is 0, order by id alone
    for K in (1, 7, 40, 100):
        for mode in (1, 0):                             # mode 0 under emulation is the exact path as well
            rc, ids, sc, _, _ = sim_call("emu", table, qids, K, metric, mode)
            assert rc == 0
            ids_o, sc_o = similar_reference(table, qids, K, metric)
            assert_same(ids, sc, ids_o, sc_o, (K, mode))
        for u, q in enumerate(qids):
            live = ids[u][np.isfinite(sc[u])]
            assert q not in ids[u] and 0 not in live and len(live) == min(K, V - 2)
    assert (ids[:, V - 2:] == 0).all() and np.isneginf(sc[:, V - 2:]).all()    # K > V - 2 eligible items: padded
    if metric == "cosine":
        assert (ids[qids.index(40), :V - 2] == np.setdiff1d(np.arange(1, V), [40])).all()
        assert not np.isnan(sc).any()


@pytest.mark.emu
def test_item_rows_gather_and_normalisation_emulated():
    lib, dev = backend("emu")
    rng = np.random.RandomState(4)
    V, H = 37, 20
    table = (rng.randn(V, H) * rng.choice([1e-20, 1e-3, 1.0, 1e15], (V, 1))).astype(np.float32)
    table[3] = 0.0
    table[4, :] = np.float32(1e-30)                     # every square underflows: n == 0, the zero vector
    tt = torch.from_numpy(table)
    ids = np.array([5, 0, 3, 36, -1, 37, 4, 5], np.int32)
    want = {0: table, 1: normalise(table)}
    for norm in (0, 1):
        out = torch.full((len(ids), H), 9.0)
        assert lib.cast_item_rows(torch.from_numpy(ids).data_ptr(), len(ids), tt.data_ptr(), None, 0, V, H, norm,
                                  out.data_ptr(), None) == 0
        exp = np.where(((ids >= 0) & (ids < V))[:, None], want[norm][np.clip(ids, 0, V - 1)], 0.0).astype(np.float32)
        assert np.array_equal(out.numpy().view(np.uint32), exp.view(np.uint32)), norm
        full = torch.full((V, H), 9.0)
        assert lib.cast_item_rows(None, V, tt.data_ptr(), None, 0, V, H, norm, full.data_ptr(), None) == 0
        assert np.array_equal(full.numpy().view(np.uint32), want[norm].view(np.uint32))
    assert (normalise(table)[4] == 0).all()
    # the same rows through a row-sharded view (2 shards, cyclic, local row 0 of shard 1 a pad)
    sh = [np.zeros(((V + 1) // 2 + 1, H), np.float32) for _ in range(2)]
    sh[0][:len(table[0::2])] = table[0::2]
    sh[1][1:1 + len(table[1::2])] = table[1::2]
    sht = [torch.from_numpy(s) for s in sh]
    ptrs = torch.tensor([s.data_ptr() for s in sht], dtype=torch.int64)
    gid = np.arange(1, V, dtype=np.int32)
    for norm in (0, 1):
        out = torch.zeros(len(gid), H)
        assert lib.cast_item_rows(torch.from_numpy(gid).data_ptr(), len(gid), None, ptrs.data_ptr(), 2, V, H, norm,
                                  out.data_ptr(), None) == 0
        assert np.array_equal(out.numpy().view(np.uint32), want[norm][1:].view(np.uint32))


@pytest.mark.emu
def test_argument_validation():
    import cast_b200
    lib, dev = backend("emu")
    table = np.random.RandomState(2).randn(50, 8).astype(np.float32)
    assert lib.cast_similar_items_workspace_bytes(3, 50, 8, 0, COSINE) == 0
    assert lib.cast_similar_items_workspace_bytes(3, 50, 8, 257, DOT) == 0
    assert lib.cast_similar_items_workspace_bytes(3, 50, 8, 5, 2) == 0
    assert lib.cast_similar_items_workspace_bytes(3, 50, 8, 5, COSINE) > lib.cast_similar_items_workspace_bytes(
        3, 50, 8, 5, DOT) > lib.cast_topk_full_workspace_bytes(3, 50, 8, 5)
    assert sim_call("emu", table, [1, 2, 3], 0, "dot", ws_bytes=1 << 20)[0] == ERR_BAD_ARG
    assert sim_call("emu", table, [1, 2, 3], 257, "dot", ws_bytes=1 << 20)[0] == ERR_BAD_ARG
    assert b"K must be" in lib.cast_last_error_string()
    assert sim_call("emu", table, [1, 2, 3], 5, 2, ws_bytes=1 << 20)[0] == ERR_BAD_ARG
    assert b"metric" in lib.cast_last_error_string()
    need = lib.cast_similar_items_workspace_bytes(3, 50, 8, 5, COSINE)
    assert sim_call("emu", table, [1, 2, 3], 5, "cosine", ws_bytes=need - 1)[0] == ERR_WORKSPACE
    assert sim_call("emu", table, [1, 2, 3], 256, "cosine")[0] == 0
    args = make_args(hidden_units=8, maxlen=6, num_heads=1, num_blocks=1)
    m = cast_b200.SASRec(10, 40, args, device=dev, _lib=lib, use_graph=False, seed=1)
    for bad in ([0], [41], [1, -3], [1.5]):
        with pytest.raises(ValueError, match="query ids"):
            m.similar_items(bad, 5)
    for k in (0, 257):
        with pytest.raises(ValueError, match="k must be"):
            m.similar_items([1], k)
    with pytest.raises(ValueError, match="metric"):
        m.similar_items([1], 5, "l2")
    ids, sc = m.similar_items([40, 1], 256, "dot")
    assert ids.shape == (2, 256) and (ids[:, 39:] == 0).all() and np.isneginf(sc[:, 39:]).all()
    assert m.similar_items([], 3)[0].shape == (0, 3)


def _item_table(m):
    return m.state_dict()["item_emb"].numpy()


@pytest.mark.emu
@pytest.mark.parametrize("metric", ["cosine", "dot"])
def test_model_similar_items_emulated(metric):
    import cast_b200
    from cast_b200 import evaluation as cev
    lib, dev = backend("emu")
    args = make_args(hidden_units=12, maxlen=10, num_heads=1, num_blocks=1, dropout_rate=0.0)
    m = cast_b200.SASRec(80, 300, args, device=dev, _lib=lib, use_graph=False, seed=3)
    table = _item_table(m)
    qids = [300, 1, 7, 150, 7]
    ids, sc = m.similar_items(qids, 10, metric)
    assert ids.dtype == np.int32 and sc.dtype == np.float32
    assert_same(ids, sc, *similar_reference(table, qids, 10, metric))
    assert_same(*m.similar_items(qids, 10, metric, mode=1), ids, sc, "mode 1")
    items, nbr, scs = cev.similar_items_all(m, 4, batch=64, lo=250, metric=metric)
    assert (items == np.arange(251, 301)).all()
    assert_same(nbr, scs, *similar_reference(table, items, 4, metric))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _sharded_worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    import cast_b200
    from cast_b200 import dist as cdist
    cdist.init_from_env("gloo")
    lib, dev = backend("emu")
    T, H, V = 10, 12, 301
    args = make_args(hidden_units=H, maxlen=T, num_heads=1, num_blocks=1, dropout_rate=0.0)
    arena = cdist.PeerArena(lib, dev)
    m = cast_b200.SASRec(80, V, args, device=dev, _lib=lib, use_graph=False, seed=3, item_shard=(rank, world),
                         alloc=arena.alloc)
    cdist.attach(m.engine, arena=arena)
    qids = np.array([1, 2, 3, 150, 300, 301, 64, 2], np.int32)      # both owners, the last id, a repeated query
    per = len(qids) // world
    sl = slice(rank * per, (rank + 1) * per)
    parts = [None] * world
    res = [m.similar_items(qids[sl], k, metric, mode=mode) for metric in ("cosine", "dot")
           for k, mode in ((12, 1), (5, 0), (256, 0))]
    dist.all_gather_object(parts, res)
    if rank == 0:
        single = cast_b200.SASRec(80, V, args, device=dev, _lib=lib, use_graph=False, seed=3)
        torch.save({"sharded": [np.concatenate([p[i][j] for p in parts]) for i in range(len(res)) for j in (0, 1)],
                    "single": [a for metric in ("cosine", "dot") for k, mode in ((12, 1), (5, 0), (256, 0))
                               for a in single.similar_items(qids, k, metric, mode=mode)],
                    "table": _item_table(single), "qids": qids}, out)
    dist.barrier()
    arena.close()
    dist.destroy_process_group()


@pytest.mark.emu
def test_similar_items_item_sharded_equals_single_process(tmp_path):
    """row-sharded item table over 2 ranks (gloo): query rows read from their owners, per-shard top k with the query's
    own row excluded where the shard holds it, merge by (score desc, id asc) — bits equal to the single-process call"""
    out = str(tmp_path / "res.pt")
    mp.spawn(_sharded_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    r = torch.load(out, weights_only=False)
    for a, b in zip(r["sharded"], r["single"]):
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
    assert_same(r["single"][0], r["single"][1], *similar_reference(r["table"], r["qids"], 12, "cosine"))
    assert (r["single"][0] > 0).all()


@pytest.mark.emu
def test_main_driver_similar_items_writes_npz(tmp_path, monkeypatch):
    import main as driver
    lib, dev = backend("emu")
    argv = ["--dataset", DATASET, "--train_dir", "unit", "--model", "sasrec", "--maxlen", "8", "--hidden_units", "12",
            "--batch_size", "16", "--num_epochs", "1", "--dropout_rate", "0.2", "--bin_in_hours", "48",
            "--eval_every", "1", "--eval_batch", "40", "--model_path", str(tmp_path)]
    assert driver.run(driver.build_parser().parse_args(argv), device=dev, lib=lib) == 0
    run_dir = os.path.join(str(tmp_path), "ref_dataset.txt")
    (sub,) = os.listdir(run_dir)
    d = os.path.join(run_dir, sub)
    seen = {}
    orig = driver.write_similar_items

    def keep(model, args, rank, world):      # the model as the driver left it (it trains one step before testing)
        seen["model"] = model
        return orig(model, args, rank, world)

    monkeypatch.setattr(driver, "write_similar_items", keep)
    for metric in ("dot", "cosine"):
        args = driver.build_parser().parse_args(argv + ["--test_model", d, "--test_seq_len", "3", "--similar_items",
                                                        "5", "--similarity", metric])
        assert driver.run(args, device=dev, lib=lib) == 0
        r = np.load(os.path.join(d, "similar_items_top5.npz"))
        m = seen.pop("model")
        assert (r["items"] == np.arange(1, m.itemnum + 1)).all()
        assert r["neighbours"].shape == (m.itemnum, 5) and r["scores"].dtype == np.float32
        ids, sc = m.similar_items(r["items"], 5, metric)
        assert_same(r["neighbours"], r["scores"], ids, sc, metric)
        assert not (r["neighbours"] == r["items"][:, None]).any()


# ------------------------------------------------------------------------------------------------ B200
def _case(V, H, metric):
    U = 48
    rng = np.random.RandomState(V + H)
    qids = np.concatenate([[1, V - 1], rng.choice(np.arange(2, V - 1), U - 2, replace=False)]).astype(np.int32)
    table = make_table(V, H, V * 7 + H, ties_for=qids[:6], K=10, zero_rows=5, parallel=20)
    ids_o, sc_o = similar_reference(table, qids, 256, metric)
    return table, qids, ids_o, sc_o


@pytest.mark.gpu
@pytest.mark.parametrize("metric", ["cosine", "dot"])
@pytest.mark.parametrize("V,H", [(3417, 50), (5000, 64), (1025, 128), (100003, 256)])
def test_similar_items_both_modes_match_numpy_gpu(V, H, metric):
    table, qids, ids_o, sc_o = _case(V, H, metric)
    for K in (1, 10, 100, 256):
        for mode in (1, 0):
            rc, ids, sc, stats, flag = sim_call("gpu", table, qids, K, metric, mode)
            assert rc == 0 and flag == 0, (K, mode, rc, flag)
            assert_same(ids, sc, ids_o[:, :K], sc_o[:, :K], (K, mode))     # the top K is the prefix of the top 256
        if V >= 100000:
            assert stats[1] == 0                                            # large catalogs: no fallback


@pytest.mark.gpu
@pytest.mark.parametrize("metric", ["cosine", "dot"])
def test_similar_items_tied_block_forces_fallback_gpu(metric):
    rng = np.random.RandomState(6)
    V, H, K = 20000, 64, 100
    table = (rng.randn(V, H) * 0.3).astype(np.float32)
    qids = np.array([7, 8, 9, 10], np.int32)
    s = similar_scores(table, qids[:1], metric)[0]
    s[[0, 7]] = -np.inf
    b = int(np.argsort(-s)[K // 2])
    blk = rng.choice(np.setdiff1d(np.arange(1, V), [b, *qids]), 3000, replace=False)
    table[blk] = table[b]             # 3001 identical rows tied at query 7's K boundary: more than the buffer holds
    ids_o, sc_o = similar_reference(table, qids, K, metric)
    for mode in (1, 0):
        rc, ids, sc, stats, flag = sim_call("gpu", table, qids, K, metric, mode)
        assert rc == 0 and flag == 0
        assert_same(ids, sc, ids_o, sc_o, mode)
    assert stats[1] > 0, "the tied block must overflow the candidate buffer"
    assert np.isin(ids_o[0], blk).sum() > 10


@pytest.mark.gpu
def test_similar_items_parallel_rows_cosine_gpu():
    """rows c * e of one direction with different c: their normalised bits may or may not coincide; the tensor-core
    filter and brute force must agree with the restatement either way"""
    rng = np.random.RandomState(8)
    V, H, K = 4097, 128, 64
    table = (rng.randn(V, H) * 0.3).astype(np.float32)
    base = table[11].copy()
    grp = rng.choice(np.arange(12, V), 200, replace=False)
    table[grp] = base * rng.uniform(1e-3, 1e3, 200).astype(np.float32)[:, None]
    qids = np.array([11, int(grp[0]), 2, 3], np.int32)
    ids_o, sc_o = similar_reference(table, qids, K, "cosine")
    assert np.isin(ids_o[0], grp).all()
    for mode in (1, 0):
        rc, ids, sc, _, flag = sim_call("gpu", table, qids, K, "cosine", mode)
        assert rc == 0 and flag == 0
        assert_same(ids, sc, ids_o, sc_o, mode)


@pytest.mark.gpu
@pytest.mark.parametrize("metric", ["cosine", "dot"])
def test_similar_items_deterministic_and_batch_independent_gpu(metric):
    V, H, K = 30001, 128, 50
    rng = np.random.RandomState(9)
    table = make_table(V, H, 9, zero_rows=3, parallel=10)
    qids = rng.randint(1, V, 513).astype(np.int32)
    _, ids_a, sc_a, _, _ = sim_call("gpu", table, qids, K, metric)
    _, ids_b, sc_b, _, _ = sim_call("gpu", table, qids, K, metric)
    assert np.array_equal(ids_a, ids_b) and np.array_equal(sc_a.view(np.uint32), sc_b.view(np.uint32))
    for u in (0, 200, 512):
        _, ids1, sc1, _, _ = sim_call("gpu", table, qids[u:u + 1], K, metric)
        assert np.array_equal(ids1[0], ids_a[u]) and np.array_equal(sc1[0].view(np.uint32), sc_a[u].view(np.uint32))
    _, ids2, sc2, _, _ = sim_call("gpu", table, np.concatenate([qids[200:260], qids[:7]]), K, metric)
    assert_same(ids2[:60], sc2[:60], ids_a[200:260], sc_a[200:260])


@pytest.mark.gpu
@pytest.mark.parametrize("model_name", ["sasrec", "cast_3"])
def test_similar_items_model_level_gpu(model_name):
    """after graph-mode training steps: the call equals the restatement on state_dict(), and a call between two steps
    changes neither the parameters / Adam moments nor the next step's bits"""
    import cast_b200
    B, T, V = 32, 20, 700
    args = make_args(hidden_units=64, maxlen=T, num_heads=1, num_blocks=2, dropout_rate=0.2)
    batches = [synth_batch(B, T, V, seed=s) for s in range(4)]

    def step(m, b):
        m.train_step(b["u"], b["seq"], b["pos"], b["neg"], b["timeseq"], b["hours"], b["days"])

    ms = [cast_b200.build_model(model_name, 100, V, 5, args, seed=5) for _ in range(2)]
    for m in ms:
        assert m.use_graph
        for b in batches[:3]:
            step(m, b)
    m, ref = ms
    eng = m.engine
    before = [t.clone() for t in (eng.w, eng.m, eng.v, eng.adam_state)]
    table = _item_table(m)
    qids = np.arange(1, V + 1, dtype=np.int32)
    for metric in ("cosine", "dot"):
        ids, sc = m.similar_items(qids, 10, metric)
        assert_same(ids, sc, *similar_reference(table, qids, 10, metric), metric)
        assert_same(*m.similar_items(qids, 10, metric, mode=1), ids, sc, "mode 1")
    for a, b in zip(before, (eng.w, eng.m, eng.v, eng.adam_state)):
        assert torch.equal(a, b)
    step(m, batches[3])
    step(ref, batches[3])
    for a, b in zip((eng.w, eng.m, eng.v), (ref.engine.w, ref.engine.m, ref.engine.v)):
        assert torch.equal(a, b)
