"""Per-item score offsets (`item_bias`) on exact top-K recommendation and item-to-item retrieval
(`cast_topk_full_biased`, `cast_similar_items_biased`, `Model.recommend` / `Model.similar_items(..., item_bias=)`):
ids and score bits against the numpy restatement of the contract, `biased_reference` below — scores
(canonical_logits + b).astype(float32), eligible items j in [1, V) with b_j != -inf that are not excluded (and not the
query), order by score descending then id ascending, (0, -inf) padding.  The tensor-core filter (mode 0) must return
the bits of brute force (mode 1) for every kind of bias: random, popularity correction, deny lists, dense and sparse
allow lists, allow lists smaller than K, and large offsets that turn whole groups of items into exact ties."""
import ctypes
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from helpers import O, backend, golden_batch, make_args, synth_batch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DATASET = os.path.join(ROOT, "tests", "golden", "ref_dataset.txt")
ERR_BAD_ARG = -1
DOT, COSINE = 0, 1
METRIC = {"dot": DOT, "cosine": COSINE}
NINF = np.float32(-np.inf)


# ------------------------------------------------------------------------------------------------ restatement
def normalise(table):
    """canonical row normalisation of similar_items: n = sqrt_rn(k-ascending, separately rounded sum of squares)"""
    e = np.asarray(table, np.float32)
    n2 = np.zeros(e.shape[0], np.float32)
    for k in range(e.shape[1]):
        n2 = (n2 + (e[:, k] * e[:, k]).astype(np.float32)).astype(np.float32)
    n = np.sqrt(n2).astype(np.float32)
    out = np.zeros_like(e)
    nz = n != 0
    out[nz] = (e[nz] / n[nz, None]).astype(np.float32)
    return out


def biased_reference(logits, bias, K, exclude=None):
    """logits [U, V] canonical scores; bias [V] float32 (entry 0 ignored); exclude: per row, ids to leave out"""
    s = (logits + np.asarray(bias, np.float32)[None, :]).astype(np.float32)
    U, V = s.shape
    ids = np.zeros((U, K), np.int32)
    sc = np.full((U, K), NINF, np.float32)
    for u in range(U):
        ok = np.asarray(bias, np.float32) != NINF
        ok[0] = False
        if exclude is not None:
            r = np.asarray(list(exclude[u]), np.int64)
            ok[r[(r >= 0) & (r < V)]] = False
        j = np.flatnonzero(ok)
        o = j[np.lexsort((j, -s[u, j]))][:K]
        ids[u, :len(o)] = o
        sc[u, :len(o)] = s[u, o]
    return ids, sc


def similar_logits(table, qids, metric):
    rows = normalise(table) if metric == "cosine" else np.asarray(table, np.float32)
    return O.canonical_logits(rows[np.asarray(qids)], rows)


def assert_same(ids, sc, ids_o, sc_o, what=""):
    bad = np.flatnonzero((ids != ids_o).any(1) | (sc.view(np.uint32) != sc_o.view(np.uint32)).any(1))
    assert bad.size == 0, (what, bad[:8], ids[bad[:1]], ids_o[bad[:1]], sc[bad[:1]], sc_o[bad[:1]])


def csr(lists):
    ptr = np.zeros(len(lists) + 1, np.int32)
    flat = []
    for u, r in enumerate(lists):
        ids = np.sort(np.asarray(list(r), np.int64))
        flat.append(ids)
        ptr[u + 1] = ptr[u] + len(ids)
    return ptr, np.concatenate(flat + [np.zeros(1, np.int64)]).astype(np.int32)


def _stream(dev):
    return torch.cuda.current_stream(dev).cuda_stream if dev.type == "cuda" else None


def topk_call(kind, users, table, K, bias, exclude=None, mode=0):
    """cast_topk_full_biased (bias None -> a null pointer); returns (rc, ids, scores, stats, watchdog flag)"""
    lib, dev = backend(kind)
    U, H = users.shape
    V = table.shape[0]
    tu = torch.from_numpy(np.ascontiguousarray(users, np.float32)).to(dev)
    tt = torch.from_numpy(np.ascontiguousarray(table, np.float32)).to(dev)
    tb = None if bias is None else torch.from_numpy(np.ascontiguousarray(bias, np.float32)).to(dev)
    ep = ei = None
    if exclude is not None:
        p, i = csr(exclude)
        ep, ei = torch.from_numpy(p).to(dev), torch.from_numpy(i).to(dev)
    ids = torch.full((U, K), -7, dtype=torch.int32, device=dev)
    sc = torch.full((U, K), 7.0, dtype=torch.float32, device=dev)
    stats = torch.zeros(2, dtype=torch.int64, device=dev)
    wsb = lib.cast_topk_full_workspace_bytes(U, V, H, K)
    ws = torch.empty(wsb // 4 + 16, dtype=torch.int32, device=dev)
    p_ = lambda t: None if t is None else t.data_ptr()  # noqa: E731
    rc = lib.cast_topk_full_biased(tu.data_ptr(), H, tt.data_ptr(), V, H, U, K, p_(ep), p_(ei), p_(tb), mode,
                                   ids.data_ptr(), sc.data_ptr(), stats.data_ptr(), ws.data_ptr(), wsb, _stream(dev))
    flag = ctypes.c_int(-1)
    if rc == 0:
        assert lib.cast_topk_full_status(ws.data_ptr(), U, V, H, K, ctypes.byref(flag), _stream(dev)) == 0
    return rc, ids.cpu().numpy(), sc.cpu().numpy(), stats.cpu().numpy(), flag.value


def sim_call(kind, table, qids, K, metric, bias, mode=0):
    """cast_similar_items_biased on a replicated table, each query's own row excluded"""
    lib, dev = backend(kind)
    V, H = table.shape
    U = len(qids)
    m = METRIC[metric]
    tt = torch.from_numpy(np.ascontiguousarray(table, np.float32)).to(dev)
    tb = None if bias is None else torch.from_numpy(np.ascontiguousarray(bias, np.float32)).to(dev)
    q = torch.from_numpy(np.asarray(qids, np.int32)).to(dev)
    ep = torch.arange(U + 1, dtype=torch.int32).to(dev)
    ids = torch.full((U, K), -7, dtype=torch.int32, device=dev)
    sc = torch.full((U, K), 7.0, dtype=torch.float32, device=dev)
    stats = torch.zeros(2, dtype=torch.int64, device=dev)
    wsb = lib.cast_similar_items_workspace_bytes(U, V, H, K, m)
    ws = torch.empty(wsb // 4 + 16, dtype=torch.int32, device=dev)
    rc = lib.cast_similar_items_biased(q.data_ptr(), U, tt.data_ptr(), V, None, 0, V, H, K, m, ep.data_ptr(),
                                       q.data_ptr(), None if tb is None else tb.data_ptr(), mode, ids.data_ptr(),
                                       sc.data_ptr(), stats.data_ptr(), ws.data_ptr(), wsb, _stream(dev))
    flag = ctypes.c_int(-1)
    if rc == 0:
        assert lib.cast_similar_items_status(ws.data_ptr(), U, V, H, K, ctypes.byref(flag), _stream(dev)) == 0
    return rc, ids.cpu().numpy(), sc.cpu().numpy(), stats.cpu().numpy(), flag.value


def make_bias(kind, V, seed, K=10):
    """float32 [V] biases: 'zero', 'random', 'popularity' (-a log(1 + c_j), seeded Zipf counts), 'deny' (random
    removals), 'allow90' / 'allow1' (allow lists of 90 % / 1 % of the items), 'allow_lt_k' (fewer items than K),
    'ties' (a +1e8 offset on a group of items: their scores collapse to one value, ids decide), 'mixed'"""
    rng = np.random.RandomState(seed)
    b = np.zeros(V, np.float32)
    if kind == "random":
        b = (rng.randn(V) * 0.5).astype(np.float32)
    elif kind == "popularity":
        counts = rng.zipf(1.3, V).clip(0, 10 ** 6)
        b = (-0.3 * np.log1p(counts)).astype(np.float32)
    elif kind == "deny":
        b[rng.rand(V) < 0.3] = NINF
    elif kind in ("allow90", "allow1"):
        keep = rng.rand(V) < (0.9 if kind == "allow90" else 0.01)
        keep[rng.randint(1, V)] = True
        b[~keep] = NINF
    elif kind == "allow_lt_k":
        b[:] = NINF
        b[rng.choice(np.arange(1, V), max(1, K // 2), replace=False)] = 0.0
    elif kind == "ties":
        b[rng.choice(np.arange(1, V), min(V - 1, 3 * K + 7), replace=False)] = np.float32(1e8)
    elif kind == "mixed":
        b = (rng.randn(V) * 0.2).astype(np.float32)
        b[rng.rand(V) < 0.2] = NINF
        b[rng.choice(np.arange(1, V), min(V - 1, K), replace=False)] = np.float32(3e7)
    b[0] = np.float32(rng.randn())              # entry 0 is ignored whatever it holds
    return b


KINDS = ["zero", "random", "popularity", "deny", "allow90", "allow1", "allow_lt_k", "ties", "mixed"]


def make_users_table(U, V, H, seed):
    rng = np.random.RandomState(seed)
    table = (rng.randn(V, H) * 0.3).astype(np.float32)
    users = (rng.randn(U, H) * 0.5).astype(np.float32)
    table[rng.randint(1, V, 4)] = table[rng.randint(1, V)]          # duplicated rows: exact ties in the logits too
    exclude = [set(rng.randint(1, V, rng.randint(0, 12)).tolist()) for _ in range(U)]
    return users, table, exclude


# ------------------------------------------------------------------------------------------------ host emulation
@pytest.mark.emu
@pytest.mark.parametrize("kind", KINDS)
def test_topk_biased_emulated(kind):
    U, V, H = 6, 301, 12
    users, table, exclude = make_users_table(U, V, H, 1)
    users[5] = 0.0                                                  # every logit +0: bias and id decide alone
    bias = make_bias(kind, V, 2, K=10)
    logits = O.canonical_logits(users, table)
    for K in (1, 10, 40):
        for excl in (None, exclude):
            ids_o, sc_o = biased_reference(logits, bias, K, excl)
            for mode in (1, 0):                                     # mode 0 under emulation is the exact path as well
                rc, ids, sc, _, _ = topk_call("emu", users, table, K, bias, excl, mode)
                assert rc == 0
                assert_same(ids, sc, ids_o, sc_o, (K, mode, excl is None))
            eligible = (bias[1:] != NINF).sum()
            assert (ids[:, min(K, eligible):] == 0).all() or excl is not None
            assert not np.isin(ids[ids > 0], np.flatnonzero(bias == NINF)).any()
    if kind == "ties":            # user 5's scores are the offsets: the boosted group fills its list in id order
        ids_t, sc_t = biased_reference(logits, bias, 40)
        grp = np.flatnonzero(bias[1:] == np.float32(1e8)) + 1
        assert (ids_t[5, :len(grp)] == grp).all() and (sc_t[5, :len(grp)] == np.float32(1e8)).all()
    if kind == "allow_lt_k":
        assert (ids[:, 5:] == 0).all() and np.isneginf(sc[:, 5:]).all()


@pytest.mark.emu
def test_zero_bias_returns_the_unbiased_bits_emulated():
    """canonical logits are never -0 (the sum starts at +0), so fl(s + 0) and fl(s + -0) are s bit for bit"""
    users, table, exclude = make_users_table(5, 200, 16, 3)
    users[4] = 0.0
    rc, ids, sc, _, _ = topk_call("emu", users, table, 30, None, exclude)
    assert rc == 0
    for z in (0.0, -0.0):
        rc, ids_z, sc_z, _, _ = topk_call("emu", users, table, 30, np.full(200, z, np.float32), exclude)
        assert rc == 0 and np.array_equal(ids, ids_z) and (sc == sc_z).all()
        assert np.array_equal(sc.view(np.uint32), sc_z.view(np.uint32))


@pytest.mark.emu
@pytest.mark.parametrize("metric", ["cosine", "dot"])
def test_similar_items_biased_emulated(metric):
    rng = np.random.RandomState(4)
    V, H = 150, 12
    table = (rng.randn(V, H) * 0.3).astype(np.float32)
    table[rng.randint(1, V, 5)] = 0.0
    qids = [1, 5, 17, 33, 149, 40, 5]
    for kind in ("random", "popularity", "deny", "allow_lt_k", "ties"):
        bias = make_bias(kind, V, 5, K=8)
        bias[5] = np.float32(1e9)                   # query 5's own huge boost must not bring it back
        logits = similar_logits(table, qids, metric)
        excl = [[q] for q in qids]
        for K in (1, 8, 60):
            ids_o, sc_o = biased_reference(logits, bias, K, excl)
            for mode in (1, 0):
                rc, ids, sc, _, _ = sim_call("emu", table, qids, K, metric, bias, mode)
                assert rc == 0
                assert_same(ids, sc, ids_o, sc_o, (kind, K, mode))
            assert not (ids == np.asarray(qids)[:, None]).any()


@pytest.mark.emu
def test_misaligned_bias_is_rejected():
    lib, dev = backend("emu")
    U, V, H, K = 2, 50, 8, 5
    users = torch.zeros(U, H)
    table = torch.zeros(V, H)
    b = torch.zeros(V + 4)
    out_i, out_s = torch.zeros(U, K, dtype=torch.int32), torch.zeros(U, K)
    wsb = lib.cast_topk_full_workspace_bytes(U, V, H, K)
    ws = torch.empty(wsb // 4 + 16, dtype=torch.int32)
    rc = lib.cast_topk_full_biased(users.data_ptr(), H, table.data_ptr(), V, H, U, K, None, None, b.data_ptr() + 4, 0,
                                   out_i.data_ptr(), out_s.data_ptr(), None, ws.data_ptr(), wsb, None)
    assert rc == ERR_BAD_ARG and b"aligned" in lib.cast_last_error_string()
    q = torch.ones(U, dtype=torch.int32)
    wsb = lib.cast_similar_items_workspace_bytes(U, V, H, K, DOT)
    ws = torch.empty(wsb // 4 + 16, dtype=torch.int32)
    rc = lib.cast_similar_items_biased(q.data_ptr(), U, table.data_ptr(), V, None, 0, V, H, K, DOT, None, None,
                                       b.data_ptr() + 4, 0, out_i.data_ptr(), out_s.data_ptr(), None, ws.data_ptr(),
                                       wsb, None)
    assert rc == ERR_BAD_ARG and b"aligned" in lib.cast_last_error_string()


def _sasrec(lib, dev, V=300, H=12, T=10, **kw):
    import cast_b200
    args = make_args(hidden_units=H, maxlen=T, num_heads=1, num_blocks=1, dropout_rate=0.0)
    return cast_b200.SASRec(80, V, args, device=dev, _lib=lib, use_graph=False, seed=3, **kw)


def _model_last(m, B):
    eng = m.engine
    last = eng.ctx(B).seq_emb.view(B, eng.T, eng.H)[:, -1, :].cpu().numpy()
    table = eng.P["item_emb"].cpu().numpy().copy()
    table[0] = 0
    return last, table


@pytest.mark.emu
def test_item_bias_validation():
    from cast_b200.models import check_item_bias
    lib, dev = backend("emu")
    m = _sasrec(lib, dev, V=40)
    gb = {"seq": np.random.RandomState(0).randint(0, 41, (2, 10)).astype(np.int32)}
    ok = np.zeros(41, np.float32)
    for bad, what in ((np.full(41, np.nan), "NaN"), (np.r_[ok[:7], np.inf, ok[8:]], "+inf"),
                      (np.full(41, 1e39), "float64 that rounds to +inf"), (np.r_[np.nan, ok[1:]], "NaN at entry 0")):
        for arr in (bad, torch.from_numpy(np.asarray(bad))):
            with pytest.raises(ValueError, match="NaN or"):
                m.recommend(gb["seq"], 5, item_bias=arr)
            with pytest.raises(ValueError, match="NaN or"):
                m.similar_items([1, 2], 5, item_bias=arr)
    for bad in (np.zeros(40), np.zeros(42), np.zeros((41, 1)), torch.zeros(2, 41)):
        with pytest.raises(ValueError, match="shape"):
            m.recommend(gb["seq"], 5, item_bias=bad)
        with pytest.raises(ValueError, match="shape"):
            m.similar_items([3], 5, item_bias=bad)
    for bad in (np.zeros(41, bool), np.zeros(41, np.complex64), np.array(["a"] * 41), torch.zeros(41, dtype=torch.bool)):
        with pytest.raises(ValueError, match="real"):
            check_item_bias(bad, 40)
    other = _sasrec(lib, dev, V=40)
    with pytest.raises(ValueError, match="another model"):
        m.recommend(gb["seq"], 5, item_bias=other.prepare_item_bias(ok))
    # accepted: numpy of any real dtype, torch tensors, -inf, a prepared ItemBias; rounded once to float32
    b64 = np.random.RandomState(1).randn(41) * 1e-3 + 1.0
    b64[3] = -np.inf
    ids, sc = m.recommend(gb["seq"], 5, item_bias=b64)
    for same in (b64.astype(np.float32), torch.from_numpy(b64), m.prepare_item_bias(b64)):
        ids2, sc2 = m.recommend(gb["seq"], 5, item_bias=same)
        assert_same(ids2, sc2, ids, sc)
    assert 3 not in ids
    assert m.recommend(gb["seq"], 5, item_bias=np.arange(41))[0].shape == (2, 5)
    assert m.prepare_item_bias(None) is None


@pytest.mark.emu
def test_model_recommend_and_similar_items_biased_emulated():
    from cast_b200 import evaluation as cev
    lib, dev = backend("emu")
    m = _sasrec(lib, dev)
    B = 8
    gb = golden_batch(B=B, T=10)
    excl = [set(int(i) for i in gb["seq"][u] if i > 0) for u in range(B)]
    for kind in ("popularity", "mixed", "allow_lt_k"):
        bias = make_bias(kind, 301, 7, K=10)
        ids, sc = m.recommend(gb["seq"], 10, excl, item_bias=bias)
        last, table = _model_last(m, B)
        assert_same(ids, sc, *biased_reference(O.canonical_logits(last, table), bias, 10, excl), kind)
        assert_same(*m.recommend(gb["seq"], 10, excl, mode=1, item_bias=torch.from_numpy(bias)), ids, sc, "mode 1")
        for metric in ("cosine", "dot"):
            items, nbr, scs = cev.similar_items_all(m, 6, batch=64, lo=230, metric=metric, item_bias=bias)
            assert (items == np.arange(231, 301)).all()
            ref = biased_reference(similar_logits(table, items, metric), bias, 6, [[q] for q in items])
            assert_same(nbr, scs, *ref, (kind, metric))
    # recommend_users: the bias reaches every batch, the padded tail included
    inputs = {"u": np.arange(1, 12, dtype=np.int32), "seq": golden_batch(B=11, T=10)["seq"],
              "timeseq": np.zeros((11, 10), np.int32), "hours": np.zeros((11, 10), np.int32),
              "days": np.zeros((11, 10), np.int32), "rated": [np.unique(r[r > 0]) for r in golden_batch(B=11, T=10)["seq"]]}
    bias = make_bias("deny", 301, 8)
    ids, sc = cev.recommend_users(m, inputs, 7, batch_users=4, item_bias=bias)
    for s in range(0, 11, 4):
        e = min(11, s + 4)
        want = m.recommend(inputs["seq"][s:e], 7, inputs["rated"][s:e], *(inputs[k][s:e] for k in
                                                                          ("timeseq", "hours", "days")), item_bias=bias)
        assert_same(ids[s:e], sc[s:e], *want)
    assert not np.isin(ids, np.flatnonzero(bias == NINF)).any()


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _sharded_worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    from cast_b200 import dist as cdist
    cdist.init_from_env("gloo")
    lib, dev = backend("emu")
    U, V = 8, 301
    gb = golden_batch(B=U, T=10)
    excl = [set(int(i) for i in gb["seq"][u] if i > 0) for u in range(U)]
    qids = np.array([1, 2, 3, 150, 300, 301, 64, 2], np.int32)
    biases = [make_bias(k, V + 1, 11, K=12) for k in ("popularity", "mixed", "allow_lt_k", "ties")]
    arena = cdist.PeerArena(lib, dev)
    m = _sasrec(lib, dev, V=V, item_shard=(rank, world), alloc=arena.alloc)
    cdist.attach(m.engine, arena=arena)
    per = U // world
    sl = slice(rank * per, (rank + 1) * per)

    def calls(model, rows):
        res = []
        for b in biases:
            res += [model.recommend(gb["seq"][rows], 12, excl[rows], item_bias=b, mode=mode) for mode in (0, 1)]
            res += [model.similar_items(qids[rows], 12, metric, item_bias=torch.from_numpy(b))
                    for metric in ("cosine", "dot")]
        return res

    parts = [None] * world
    dist.all_gather_object(parts, calls(m, sl))
    if rank == 0:
        single = _sasrec(lib, dev, V=V)
        torch.save({"sharded": [np.concatenate([p[i][j] for p in parts]) for i in range(len(parts[0])) for j in (0, 1)],
                    "single": [a for r in calls(single, slice(0, U)) for a in r]}, out)
    dist.barrier()
    arena.close()
    dist.destroy_process_group()


@pytest.mark.emu
def test_item_sharded_biased_equals_single_process(tmp_path):
    """row-sharded item table over 2 ranks (gloo): each rank passes b[global ids of its local rows]; the merged lists
    are the single-process lists bit for bit, for recommend and for similar_items"""
    out = str(tmp_path / "res.pt")
    mp.spawn(_sharded_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    r = torch.load(out, weights_only=False)
    assert len(r["sharded"]) == len(r["single"]) == 32
    for i, (a, b) in enumerate(zip(r["sharded"], r["single"])):
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), i


DRIVER_ARGV = ["--dataset", DATASET, "--train_dir", "unit", "--model", "sasrec", "--maxlen", "8", "--hidden_units",
               "12", "--batch_size", "16", "--num_epochs", "1", "--dropout_rate", "0.2", "--bin_in_hours", "48",
               "--eval_every", "1", "--eval_batch", "40"]


@pytest.mark.emu
def test_main_driver_item_bias(tmp_path, monkeypatch):
    import main as driver
    lib, dev = backend("emu")
    argv = DRIVER_ARGV + ["--model_path", str(tmp_path)]
    assert driver.run(driver.build_parser().parse_args(argv), device=dev, lib=lib) == 0
    run_dir = os.path.join(str(tmp_path), "ref_dataset.txt")
    (sub,) = os.listdir(run_dir)
    d = os.path.join(run_dir, sub)
    seen = {}
    orig_rec, orig_sim = driver.write_recommendations, driver.write_similar_items

    def keep_rec(model, dataset, args, rank, world):
        seen["model"] = model
        return orig_rec(model, dataset, args, rank, world)

    def keep_sim(model, args, rank, world):
        seen["model"] = model
        return orig_sim(model, args, rank, world)

    monkeypatch.setattr(driver, "write_recommendations", keep_rec)
    monkeypatch.setattr(driver, "write_similar_items", keep_sim)
    from cast_b200.data import data_partition
    from cast_b200.evaluation import build_recommend_inputs
    itemnum = data_partition(DATASET, False)[4]
    bias = make_bias("mixed", itemnum + 1, 12, K=5).astype(np.float64)
    bfile = str(tmp_path / "bias.npy")
    np.save(bfile, bias)
    test = ["--test_model", d, "--test_seq_len", "3", "--item_bias", bfile]
    args = driver.build_parser().parse_args(argv + test + ["--recommend", "5", "--similar_items", "4"])
    assert driver.run(args, device=dev, lib=lib) == 0
    m = seen.pop("model")
    denied = np.flatnonzero(bias == -np.inf)
    r = np.load(os.path.join(d, "recommendations_top5.npz"))
    assert sorted(r.files) == ["items", "scores", "users"]
    rec = build_recommend_inputs(data_partition(DATASET, False), args)
    from cast_b200.evaluation import recommend_users
    assert_same(r["items"], r["scores"], *recommend_users(m, rec, 5, 40, item_bias=bias))
    assert not np.isin(r["items"], denied).any()
    s = np.load(os.path.join(d, "similar_items_top4.npz"))
    assert sorted(s.files) == ["items", "neighbours", "scores"]
    assert_same(s["neighbours"], s["scores"], *m.similar_items(s["items"], 4, "cosine", item_bias=bias))
    assert not np.isin(s["neighbours"], denied).any()
    # rejected before any work: nothing is trained, evaluated or written
    for bad in (np.zeros(itemnum), np.r_[bias[:-1], np.inf], np.r_[np.nan, bias[1:]]):
        np.save(bfile, bad)
        for f in ("recommendations_top5.npz", "similar_items_top4.npz", "test_seq_len.txt"):
            if os.path.exists(os.path.join(d, f)):
                os.remove(os.path.join(d, f))
        with pytest.raises(ValueError):
            driver.run(args, device=dev, lib=lib)
        assert not seen and not any(os.path.exists(os.path.join(d, f)) for f in
                                    ("recommendations_top5.npz", "similar_items_top4.npz", "test_seq_len.txt"))


# ------------------------------------------------------------------------------------------------ B200
def run_both_modes(users, table, K, bias, exclude=None):
    ids_o, sc_o = biased_reference(O.canonical_logits(users, table), bias, K, exclude)
    out = {}
    for mode in (1, 0):
        rc, ids, sc, stats, flag = topk_call("gpu", users, table, K, bias, exclude, mode)
        assert rc == 0 and flag == 0, (mode, rc, flag)
        assert_same(ids, sc, ids_o, sc_o, f"mode {mode}")
        out[mode] = (ids, sc, stats)
    return out, ids_o, sc_o


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("U,V,H", [(70, 3417, 50), (129, 30001, 128), (40, 100003, 256)])
def test_topk_biased_both_modes_match_numpy_gpu(U, V, H, kind):
    users, table, exclude = make_users_table(U, V, H, U + V)
    for K in (1, 10, 100, 256):
        bias = make_bias(kind, V, V + K, K=K)
        out, ids_o, _ = run_both_modes(users, table, K, bias, exclude if K in (10, 256) else None)
        stats = out[0][2]
        eligible = int((bias[1:] != NINF).sum())
        if eligible < K:
            assert stats[1] == U and (ids_o[:, eligible:] == 0).all()     # every user on the exact path, padded
        elif V >= 30001 and kind in ("zero", "random", "popularity", "deny", "allow90"):
            assert stats[1] == 0                                            # large catalogs: no fallback
    if kind == "zero":      # the unbiased call, bit for bit
        ref = topk_call("gpu", users, table, 100, None, exclude)
        assert_same(ref[1], ref[2], *topk_call("gpu", users, table, 100, np.zeros(V, np.float32), exclude)[1:3])


@pytest.mark.gpu
def test_topk_biased_tied_block_forces_fallback_gpu():
    """a block of 3000 identical rows with one shared bias, tied at user 1's K boundary under the biased score: more
    candidates than the buffer holds, so that user takes the exact path; a -inf deny list removes user 0's best"""
    rng = np.random.RandomState(5)
    U, V, H, K = 8, 20000, 64, 100
    table = (rng.randn(V, H) * 0.3).astype(np.float32)
    users = (rng.randn(U, H) * 0.5).astype(np.float32)
    bias = make_bias("popularity", V, 6)
    approx = users.astype(np.float64) @ table.T.astype(np.float64) + bias
    approx[:, 0] = -np.inf
    bias[np.argsort(-approx[0])[:300]] = NINF
    approx[:, bias == NINF] = -np.inf
    b = int(np.argsort(-approx[1])[K // 2])
    blk = rng.choice(np.setdiff1d(np.flatnonzero(bias != NINF), [0, b]), 3000, replace=False)
    table[blk] = table[b]
    bias[blk] = bias[b]
    out, ids_o, _ = run_both_modes(users, table, K, bias)
    assert out[0][2][1] > 0, "the tied block must overflow the candidate buffer"
    assert np.isin(ids_o[1], blk).sum() > 10
    assert not np.isin(ids_o, np.flatnonzero(bias == NINF)).any()


@pytest.mark.gpu
@pytest.mark.parametrize("metric", ["cosine", "dot"])
def test_similar_items_biased_both_modes_match_numpy_gpu(metric):
    rng = np.random.RandomState(12)
    V, H = 30001, 128
    table = (rng.randn(V, H) * 0.3).astype(np.float32)
    table[rng.randint(1, V, 6)] = table[rng.randint(1, V)]
    qids = np.concatenate([[1, V - 1], rng.choice(np.arange(2, V - 1), 46, replace=False)]).astype(np.int32)
    logits = similar_logits(table, qids, metric)
    excl = [[q] for q in qids]
    for kind in ("popularity", "allow1", "allow_lt_k", "ties", "mixed"):
        for K in (1, 10, 100, 256):
            bias = make_bias(kind, V, K + 3, K=K)
            bias[qids[:4]] = np.float32(1e9)            # boosted queries: still never their own neighbour
            ids_o, sc_o = biased_reference(logits, bias, K, excl)
            for mode in (1, 0):
                rc, ids, sc, _, flag = sim_call("gpu", table, qids, K, metric, bias, mode)
                assert rc == 0 and flag == 0
                assert_same(ids, sc, ids_o, sc_o, (kind, K, mode))


@pytest.mark.gpu
def test_topk_biased_deterministic_and_batch_independent_gpu():
    U, V, H, K = 513, 30001, 128, 50
    users, table, exclude = make_users_table(U, V, H, 9)
    bias = make_bias("mixed", V, 9, K=K)
    _, ids_a, sc_a, _, _ = topk_call("gpu", users, table, K, bias, exclude)
    _, ids_b, sc_b, _, _ = topk_call("gpu", users, table, K, bias, exclude)
    assert np.array_equal(ids_a, ids_b) and np.array_equal(sc_a.view(np.uint32), sc_b.view(np.uint32))
    for u in (0, 200, 512):
        _, ids1, sc1, _, _ = topk_call("gpu", users[u:u + 1], table, K, bias, [exclude[u]])
        assert np.array_equal(ids1[0], ids_a[u]) and np.array_equal(sc1[0].view(np.uint32), sc_a[u].view(np.uint32))
    sl = list(range(200, 260)) + list(range(7))
    _, ids2, sc2, _, _ = topk_call("gpu", users[sl], table, K, bias, [exclude[u] for u in sl])
    assert_same(ids2[:60], sc2[:60], ids_a[200:260], sc_a[200:260])


@pytest.mark.gpu
@pytest.mark.parametrize("model_name", ["sasrec", "cast_3"])
def test_item_bias_model_level_gpu(model_name):
    """after graph-mode training steps: biased recommend / similar_items equal the restatement on the model's own rows,
    and the calls between two steps change neither the parameters / Adam moments nor the next step's bits"""
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
    bias = make_bias("mixed", V + 1, 13, K=10)
    b0 = batches[0]
    feats = (b0["timeseq"], b0["hours"], b0["days"])
    excl = [set(r[r > 0].tolist()) for r in b0["seq"]]
    ids, sc = m.recommend(b0["seq"], 10, excl, *feats, item_bias=bias)
    last, table = _model_last(m, B)
    assert_same(ids, sc, *biased_reference(O.canonical_logits(last, table), bias, 10, excl))
    assert_same(*m.recommend(b0["seq"], 10, excl, *feats, mode=1, item_bias=torch.from_numpy(bias).cuda()), ids, sc)
    qids = np.arange(1, V + 1, dtype=np.int32)
    for metric in ("cosine", "dot"):
        ids, sc = m.similar_items(qids, 10, metric, item_bias=bias)
        assert_same(ids, sc, *biased_reference(similar_logits(table, qids, metric), bias, 10, [[q] for q in qids]))
        assert_same(*m.similar_items(qids, 10, metric, mode=1, item_bias=bias), ids, sc, "mode 1")
    for a, b in zip(before, (eng.w, eng.m, eng.v, eng.adam_state)):
        assert torch.equal(a, b)
    step(m, batches[3])
    step(ref, batches[3])
    for a, b in zip((eng.w, eng.m, eng.v), (ref.engine.w, ref.engine.m, ref.engine.v)):
        assert torch.equal(a, b)
