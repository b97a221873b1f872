"""Exact full-catalog top-K (`cast_topk_full`, `Model.recommend`): ids and score bits against a CPU reference
(`topk_reference` below, built on `O.canonical_logits`: score descending, id ascending, (0, -inf) padding).  The
tensor-core path (mode 0) is only a filter, so it must return the same bits as the brute-force path (mode 1) on every
case: exact ties across the K boundary, near-ties inside the TF32 error band, heavy exclusions, a tied block larger
than the candidate buffer (the exact fallback), K above the number of eligible items, ragged shapes and strided user
rows."""
import ctypes
import os
import random
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from helpers import O, backend, golden_batch, make_args

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DATASET = os.path.join(ROOT, "tests", "golden", "ref_dataset.txt")
ERR_BAD_ARG, ERR_WORKSPACE = -1, -3


def topk_reference(users, table, K, exclude=None):
    """Exact full-catalog top-K on the CPU: per user the K rows j in [1,V) not in exclude[u] (ids outside [1,V)
    ignored) by canonical logit descending, then id ascending; fewer than K eligible rows pad with (0, -inf)."""
    s = O.canonical_logits(users, table)
    U, V = s.shape
    ids = np.zeros((U, K), np.int32)
    sc = np.full((U, K), -np.inf, np.float32)
    for u in range(U):
        ok = np.ones(V, bool)
        ok[0] = False
        if exclude is not None:
            r = np.asarray(list(exclude[u]), np.int64)
            ok[r[(r >= 0) & (r < V)]] = False
        j = np.flatnonzero(ok)
        o = j[np.lexsort((j, -s[u, j]))][:K]
        ids[u, :len(o)] = o
        sc[u, :len(o)] = s[u, o]
    return ids, sc


def csr(lists):
    ptr = np.zeros(len(lists) + 1, np.int32)
    flat = []
    for u, r in enumerate(lists):
        ids = np.sort(np.asarray(list(r), np.int64))      # ascending; duplicates / out-of-range ids kept on purpose
        flat.append(ids)
        ptr[u + 1] = ptr[u] + len(ids)
    return ptr, np.concatenate(flat + [np.zeros(1, np.int64)]).astype(np.int32)


def topk_call(kind, users, H, table, K, exclude=None, mode=0, ws_bytes=None):
    """users [U, ld] (first H columns used); returns (rc, ids, scores, stats, watchdog flag)"""
    lib, dev = backend(kind)
    U, ld = users.shape
    V = table.shape[0]
    tu, tt = torch.from_numpy(np.ascontiguousarray(users)).to(dev), torch.from_numpy(np.ascontiguousarray(table)).to(dev)
    ep = ei = None
    if exclude is not None:
        p, i = csr(exclude)
        ep, ei = torch.from_numpy(p).to(dev), torch.from_numpy(i).to(dev)
    kk = max(K, 1)
    ids = torch.full((U, kk), -7, dtype=torch.int32, device=dev)
    sc = torch.full((U, kk), 7.0, dtype=torch.float32, device=dev)
    stats = torch.zeros(2, dtype=torch.int64, device=dev)
    need = lib.cast_topk_full_workspace_bytes(U, V, H, K)
    wsb = need if ws_bytes is None else ws_bytes
    ws = torch.empty(max(need, wsb) // 4 + 16, dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream if dev.type == "cuda" else None
    rc = lib.cast_topk_full(tu.data_ptr(), ld, tt.data_ptr(), V, H, U, K, None if ep is None else ep.data_ptr(),
                            None if ei is None else ei.data_ptr(), mode, ids.data_ptr(), sc.data_ptr(), stats.data_ptr(),
                            ws.data_ptr(), wsb, stream)
    flag = ctypes.c_int(-1)
    if rc == 0:
        assert lib.cast_topk_full_status(ws.data_ptr(), U, V, H, K, ctypes.byref(flag), stream) == 0
    return rc, ids.cpu().numpy(), sc.cpu().numpy(), stats.cpu().numpy(), flag.value


def assert_same(ids, sc, ids_o, sc_o, what=""):
    bad = np.flatnonzero((ids != ids_o).any(1) | (sc.view(np.uint32) != sc_o.view(np.uint32)).any(1))
    assert bad.size == 0, (what, bad[:8], ids[bad[:1]], ids_o[bad[:1]], sc[bad[:1]], sc_o[bad[:1]])


def make_case(U, V, H, K, seed=0, ld_extra=0, ties=True):
    """random users / table with, for every third user, exact duplicates, a one-ulp neighbour and a 1+3e-6 neighbour
    of the row that sits near its K-th place (ties and near-ties across the K boundary)"""
    rng = np.random.RandomState(seed)
    table = (rng.randn(V, H) * 0.3).astype(np.float32)
    users = (rng.randn(U, H + ld_extra) * 0.5).astype(np.float32)
    if ties and V > 40:
        approx = users[:, :H].astype(np.float64) @ table.T.astype(np.float64)
        approx[:, 0] = -np.inf
        for u in range(0, U, 3):
            b = int(np.argsort(-approx[u])[min(K, V - 2) - 1])
            js = rng.randint(1, V, 4)
            table[js[0]] = table[b]
            table[js[1]] = table[b]
            table[js[2]] = np.nextafter(table[b], np.float32(np.inf))
            table[js[3]] = table[b] * np.float32(1 + 3e-6)
    exclude = [set(rng.randint(1, V, rng.randint(0, 12)).tolist()) for _ in range(U)]
    return users, table, exclude


# ------------------------------------------------------------------------------------------------ host emulation
@pytest.mark.emu
def test_exact_path_emulated_ties_zero_rows_padding_and_exclusions():
    rng = np.random.RandomState(1)
    V, H = 90, 12
    table = (rng.randn(V, H) * 0.3).astype(np.float32)
    table[10:14] = table[20]                         # duplicated rows: ties across the K boundary
    table[30:45] = 0.0                               # all-zero rows: many exact 0.0 ties
    users = (rng.randn(5, H + 3) * 0.5).astype(np.float32)
    users[4] = 0.0                                   # every score 0.0: order by id alone
    exclude = [[0, 3, 3, 7, 20, V + 5, 1000], [], [11, 11, 12], list(range(1, V - 3)), [-1, 0]]
    for K in (1, 7, 40):
        rc, ids, sc, _, _ = topk_call("emu", users, H, table, K, exclude, mode=1)
        assert rc == 0
        ids_o, sc_o = topk_reference(users[:, :H], table, K, exclude)
        assert_same(ids, sc, ids_o, sc_o, K)
    assert (ids[3, 3:] == 0).all() and np.isneginf(sc[3, 3:]).all()     # 3 eligible items < K: padded
    assert (ids[4] == np.arange(1, 41)).all()
    # mode 0 under emulation is the exact path as well
    rc, ids0, sc0, _, _ = topk_call("emu", users, H, table, 7, exclude, mode=0)
    ids_o, sc_o = topk_reference(users[:, :H], table, 7, exclude)
    assert rc == 0
    assert_same(ids0, sc0, ids_o, sc_o)


@pytest.mark.emu
def test_argument_validation():
    rng = np.random.RandomState(2)
    users = rng.randn(3, 8).astype(np.float32)
    table = rng.randn(50, 8).astype(np.float32)
    lib, _ = backend("emu")
    assert lib.cast_topk_full_workspace_bytes(3, 50, 8, 0) == 0
    assert lib.cast_topk_full_workspace_bytes(3, 50, 8, 257) == 0
    assert topk_call("emu", users, 8, table, 0, ws_bytes=1 << 20)[0] == ERR_BAD_ARG
    assert topk_call("emu", users, 8, table, 257, ws_bytes=1 << 20)[0] == ERR_BAD_ARG
    assert b"K must be" in lib.cast_last_error_string()
    need = lib.cast_topk_full_workspace_bytes(3, 50, 8, 5)
    assert topk_call("emu", users, 8, table, 5, ws_bytes=need - 1)[0] == ERR_WORKSPACE
    assert topk_call("emu", users, 8, table, 256)[0] == 0


def _model_last(m, B):
    eng = m.engine
    last = eng.ctx(B).seq_emb.view(B, eng.T, eng.H)[:, -1, :].cpu().numpy()
    table = eng.P["item_emb"].cpu().numpy().copy()
    table[0] = 0
    return last, table


@pytest.mark.emu
def test_recommend_emulated_golden_batch():
    import cast_b200
    lib, dev = backend("emu")
    B, T, H = 8, 10, 12
    args = make_args(hidden_units=H, maxlen=T, num_heads=1, num_blocks=1, dropout_rate=0.0)
    gb = golden_batch(B=B, T=T)
    m = cast_b200.SASRec(80, 300, args, device=dev, _lib=lib, use_graph=False, seed=3)
    excl = [set(int(i) for i in gb["seq"][u] if i > 0) for u in range(B)]
    ids, sc = m.recommend(gb["seq"], 10, excl)
    last, table = _model_last(m, B)
    ids_o, sc_o = topk_reference(last, table, 10, excl)
    assert ids.shape == (B, 10) and ids.dtype == np.int32 and sc.dtype == np.float32
    assert_same(ids, sc, ids_o, sc_o)
    ids2, sc2 = m.recommend(gb["seq"], 10)
    assert_same(ids2, sc2, *topk_reference(last, table, 10))


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
    U, T, H, V = 8, 10, 12, 300
    args = make_args(hidden_units=H, maxlen=T, num_heads=1, num_blocks=1, dropout_rate=0.0)
    gb = golden_batch(B=U, T=T)
    excl = [set(int(i) for i in gb["seq"][u] if i > 0) | {0, 299, 300, 301} for u in range(U)]
    arena = cdist.PeerArena(lib, dev)
    m = cast_b200.SASRec(80, V, args, device=dev, _lib=lib, use_graph=False, seed=3, item_shard=(rank, world),
                         alloc=arena.alloc)
    cdist.attach(m.engine, arena=arena)
    per = U // world
    sl = slice(rank * per, (rank + 1) * per)
    parts = [None] * world
    dist.all_gather_object(parts, (m.recommend(gb["seq"][sl], 12, excl[sl], mode=1), m.recommend(gb["seq"][sl], 5)))
    if rank == 0:
        single = cast_b200.SASRec(80, V, args, device=dev, _lib=lib, use_graph=False, seed=3)
        torch.save({"sharded": [np.concatenate([p[a][b] for p in parts]) for a in (0, 1) for b in (0, 1)],
                    "single": [*single.recommend(gb["seq"], 12, excl, mode=1), *single.recommend(gb["seq"], 5)]}, out)
    dist.barrier()
    arena.close()
    dist.destroy_process_group()


@pytest.mark.emu
def test_recommend_item_sharded_equals_single_process(tmp_path):
    """row-sharded item table over 2 ranks (gloo): per-shard top K, local rows -> global ids, merge by (score desc,
    id asc) — ids and score bits equal to the single-process call"""
    out = str(tmp_path / "res.pt")
    mp.spawn(_sharded_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    r = torch.load(out, weights_only=False)
    for a, b in zip(r["sharded"], r["single"]):
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
    assert (r["single"][0] > 0).all()


@pytest.mark.emu
def test_main_driver_recommend_writes_npz(tmp_path):
    import logging
    import main as driver
    from cast_b200 import data as cdata
    lib, dev = backend("emu")
    argv = ["--dataset", DATASET, "--train_dir", "unit", "--model", "sasrec", "--maxlen", "8", "--hidden_units", "12",
            "--batch_size", "16", "--num_epochs", "1", "--dropout_rate", "0.2", "--bin_in_hours", "48",
            "--eval_every", "1", "--eval_batch", "40", "--model_path", str(tmp_path)]
    assert driver.run(driver.build_parser().parse_args(argv), device=dev, lib=lib) == 0
    run_dir = os.path.join(str(tmp_path), "ref_dataset.txt")
    (sub,) = os.listdir(run_dir)
    d = os.path.join(run_dir, sub)

    class Keep(logging.Handler):
        def __init__(self):
            super().__init__()
            self.lines = []

        def emit(self, rec):
            self.lines.append(rec.getMessage())

    logs = []
    for extra in ([], ["--recommend", "5"]):
        keep = Keep()
        logger = logging.getLogger("topk_driver_test")
        logger.setLevel(logging.DEBUG)
        logger.addHandler(keep)
        args = driver.build_parser().parse_args(argv + ["--test_model", d, "--test_seq_len", "3"] + extra)
        assert driver.run(args, device=dev, lib=lib, logger=logger) == 0
        logger.removeHandler(keep)
        logs.append(keep.lines)
        assert os.path.isfile(os.path.join(d, "recommendations_top5.npz")) == bool(extra)
    assert logs[0] == logs[1]
    rows = open(os.path.join(d, "test_seq_len.txt")).read().strip().split("\n")
    assert len(rows) == 2 and rows[0] == rows[1]
    r = np.load(os.path.join(d, "recommendations_top5.npz"))
    train, valid, test, usernum = cdata.data_partition(DATASET, False)[:4]
    users, items, scores = r["users"], r["items"], r["scores"]
    assert items.shape == (len(users), 5) and scores.shape == (len(users), 5) and len(users) > 0
    for u, it in zip(users, items):
        hist = {x.item for x in list(train.get(u, [])) + list(valid.get(u, [])) + list(test.get(u, []))}
        assert not hist & set(it.tolist()), u
    assert (np.diff(scores, axis=1) <= 0).all()


# ------------------------------------------------------------------------------------------------ B200
def run_both_modes(users, H, table, K, exclude, **kw):
    ids_o, sc_o = topk_reference(users[:, :H], table, K, exclude)
    out = {}
    for mode in (1, 0):
        rc, ids, sc, stats, flag = topk_call("gpu", users, H, table, K, exclude, mode=mode, **kw)
        assert rc == 0 and flag == 0, (mode, rc, flag)
        assert_same(ids, sc, ids_o, sc_o, f"mode {mode}")
        out[mode] = (ids, sc, stats)
    return out, ids_o, sc_o


@pytest.mark.gpu
@pytest.mark.parametrize("U,V,H,K,ld_extra", [(70, 3417, 50, 10, 0), (300, 5000, 50, 100, 150), (129, 1025, 128, 1, 0),
                                              (200, 2000, 256, 256, 0), (1, 300, 50, 10, 0),
                                              (513, 30001, 128, 50, 0), (40, 100000, 256, 100, 0)])
def test_topk_both_modes_match_oracle_gpu(U, V, H, K, ld_extra):
    users, table, exclude = make_case(U, V, H, K, seed=U + V, ld_extra=ld_extra)
    out, _, sc_o = run_both_modes(users, H, table, K, exclude)
    stats = out[0][2]
    assert stats[0] >= min(K, V - 1) * U or stats[1] > 0        # at least K candidates re-scored per filtered user
    if V >= 30001:
        assert stats[1] == 0                                    # large catalogs: no user needs the fallback
        assert stats[0] <= U * (2 * K + 256)


@pytest.mark.gpu
def test_topk_adversarial_exclusions_and_tied_block_gpu():
    rng = np.random.RandomState(5)
    U, V, H, K = 8, 20000, 64, 100
    table = (rng.randn(V, H) * 0.3).astype(np.float32)
    users = (rng.randn(U, H) * 0.5).astype(np.float32)
    approx = users.astype(np.float64) @ table.T.astype(np.float64)
    approx[:, 0] = -np.inf
    order0 = np.argsort(-approx[0])
    exclude = [set(order0[:500].tolist())] + [set() for _ in range(U - 1)]     # user 0: its 500 best items excluded
    # a block of 3000 identical rows tied at user 1's K boundary: more candidates than the buffer holds -> fallback
    b = int(np.argsort(-approx[1])[K // 2])
    blk = rng.choice(np.setdiff1d(np.arange(1, V), [b]), 3000, replace=False)
    table[blk] = table[b]
    out, ids_o, _ = run_both_modes(users, H, table, K, exclude)
    assert out[0][2][1] > 0, "the tied block must overflow the candidate buffer"
    assert not set(ids_o[0].tolist()) & exclude[0]
    assert np.isin(ids_o[1], blk).sum() > 10


@pytest.mark.gpu
def test_topk_deterministic_and_batch_independent_gpu():
    U, V, H, K = 513, 30001, 128, 50
    users, table, exclude = make_case(U, V, H, K, seed=9)
    _, ids_a, sc_a, _, _ = topk_call("gpu", users, H, table, K, exclude)
    _, ids_b, sc_b, _, _ = topk_call("gpu", users, H, table, K, exclude)
    assert np.array_equal(ids_a, ids_b) and np.array_equal(sc_a.view(np.uint32), sc_b.view(np.uint32))
    for u in (0, 200, 512):
        _, ids1, sc1, _, _ = topk_call("gpu", users[u:u + 1], H, table, K, [exclude[u]])
        assert np.array_equal(ids1[0], ids_a[u]) and np.array_equal(sc1[0].view(np.uint32), sc_a[u].view(np.uint32))


@pytest.mark.gpu
@pytest.mark.parametrize("model_name", ["sasrec", "cast_3"])
def test_recommend_model_level_gpu(model_name):
    import cast_b200
    from cast_b200 import data as cdata
    from cast_b200 import evaluation as cev
    dataset = cdata.data_partition(DATASET, False)
    args = make_args(hidden_units=50, maxlen=50, num_heads=1, num_blocks=2, dropout_rate=0.2)
    args.test_model = None
    args.test_seq_len = None
    m = cast_b200.build_model(model_name, dataset[3], dataset[4], 5, args)
    p = {k: v.detach().cpu().clone() for k, v in m.engine.P.items()}
    g = torch.Generator().manual_seed(9)
    for k in p:
        if k.endswith("beta"):
            p[k] = torch.randn(p[k].shape, generator=g) * 0.2
    m.engine.load_parameters(p)
    random.seed(3)
    np.random.seed(3)
    cand = cev.build_candidates(dataset, args, "test")
    U, K = len(cand["u"]), 10
    feats = (cand["timeseq"], cand["hours"], cand["days"])
    ids, sc = m.recommend(cand["seq"], K, cand["rated"], *feats)
    last, table = _model_last(m, U)
    ids_o, sc_o = topk_reference(last, table, K, cand["rated"])
    assert_same(ids, sc, ids_o, sc_o)
    assert_same(*m.recommend(cand["seq"], K, cand["rated"], *feats, mode=1), ids_o, sc_o, "mode 1")
    logits, _, _ = m.score_candidates(cand["seq"], ids, *feats)
    assert np.array_equal(logits.view(np.uint32), sc.view(np.uint32))
    target = cand["item_idx"][:, 0]
    cgt, ceq = m.score_full_catalog(cand["seq"], target, cand["rated"], *feats)
    checked = 0
    for u in range(U):
        if ceq[u] != 0 or target[u] in set(cand["rated"][u].tolist()):
            continue
        if cgt[u] < K:
            assert ids[u, cgt[u]] == target[u], u
        else:
            assert target[u] not in ids[u], u
        checked += 1
    assert checked > U // 2
