"""optimizer="lazy_adam": tf.contrib.opt.LazyAdamOptimizer on the item table, dense TF-Adam on every other parameter.
A step updates w, m and v of the table rows its batch touches (distinct nonzero ids of seq, pos and neg) and leaves
every other row bit for bit; the gradient rows are tracked by per-row stamps against a device epoch counter, so the
table gradient needs no zeroing pass.  Host-emulated kernels (`emu`, CPU) at tiny shapes and the B200 (`gpu`)."""
import json
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from helpers import O, backend, golden_batch, make_args, oracle_batch, rel_err
from cast_b200.engine import Engine

B, T, H = 4, 10, 12
ITEMS = 300


def _engine(kind, model, optimizer, seed=5, **kw):
    lib, dev = backend(kind)
    args = make_args(**{"hidden_units": H, "maxlen": T, "num_heads": 2, "num_blocks": 1, "dropout_rate": 0.0,
                        "optimizer": optimizer, **kw})
    return Engine(model, 80, ITEMS, args, device=dev, lib=lib, seed=seed)


def _load(eng, gb, lo=0, hi=None):
    hi = gb["seq"].shape[0] if hi is None else hi
    c = eng.ctx(hi - lo)
    c.keys3.copy_(torch.from_numpy(np.stack([gb[k][lo:hi].reshape(-1) for k in ("seq", "pos", "neg")])))
    c.cids.copy_(torch.from_numpy(np.stack([gb[k][lo:hi].reshape(-1) for k in ("timeseq", "hours", "days")])))
    return c


def _batch(step):
    return golden_batch(idx=step % 3, B=B, T=T) if step < 3 else golden_batch(tag="log", idx=step % 3, B=B, T=T)


def _touched(gb, lo=0, hi=None):
    ids = np.concatenate([gb[k][lo:hi].reshape(-1) for k in ("seq", "pos", "neg")])
    return np.unique(ids[ids > 0])


def _table(eng, flat):
    return flat[:eng.P["item_emb"].numel()].reshape(eng.P["item_emb"].shape)


def _state(eng):
    return eng.w.cpu().clone(), eng.m.cpu().clone(), eng.v.cpu().clone()


@pytest.mark.emu
@pytest.mark.parametrize("model", ["sasrec", "cast_1"])
def test_first_step_equals_dense_adam(model):
    """m = v = 0: untouched rows have g = 0 and stay put under dense Adam too, so one step is the same bits"""
    gb = _batch(0)
    out = []
    for opt in ("adam", "lazy_adam"):
        eng = _engine("emu", model, opt)
        eng.launch_train_step(_load(eng, gb))
        out.append(_state(eng))
    for a, b in zip(*out):
        assert torch.equal(a, b)


class _LazyTFAdam(O.TFAdam):
    """float64 reference: TF-Adam with the item table updated on the touched rows only"""

    def step(self, params, grads, rows):
        lr_t = np.float64(np.float32(self.lr) * np.sqrt(np.float32(1) - self.b2p) / (np.float32(1) - self.b1p))
        with torch.no_grad():
            for k, w in params.items():
                sel = torch.from_numpy(rows) if k == "item_emb" else slice(None)
                g, m, v = grads[k][sel], self.m[k][sel], self.v[k][sel]
                m = self.b1 * m + (1 - self.b1) * g
                v = self.b2 * v + (1 - self.b2) * g * g
                w[sel] = w[sel] - lr_t * m / (v.sqrt() + self.eps)
                self.m[k][sel], self.v[k][sel] = m, v
        self.b1p = np.float32(self.b1p * np.float32(self.b1))
        self.b2p = np.float32(self.b2p * np.float32(self.b2))


@pytest.mark.emu
@pytest.mark.parametrize("model", ["sasrec", "cast_4"])
def test_steps_track_lazy_reference(model):
    """K = 4 steps on reference-sampler batches against the oracle's gradients + float64 lazy TF-Adam: w, m and v within
    1e-4 relative; rows a step does not touch are bit-identical before and after it; row 0 never changes."""
    eng = _engine("emu", model, "lazy_adam")
    args = eng.args
    # beta != 0: with beta = 0 the reference's query mask sign(|sum_H LN(x)|) is decided by rounding noise (DESIGN.md)
    g = torch.Generator().manual_seed(3)
    eng.load_parameters({k: torch.randn(v.shape, generator=g) * 0.1 for k, v in eng.P.items() if k.endswith("beta")})
    p = {k: v.detach().cpu().double().clone() for k, v in eng.P.items()}
    ref = _LazyTFAdam(p, lr=args.lr)
    w0 = _state(eng)
    for step in range(4):
        gb = _batch(step)
        rows = _touched(gb)
        before = _state(eng)
        eng.launch_train_step(_load(eng, gb))
        after = _state(eng)
        _, _, grads = O.train_step(model, {k: v.float() for k, v in p.items()}, None, args, oracle_batch(gb))
        ref.step(p, {k: g.double() for k, g in grads.items()}, rows)
        keep = np.setdiff1d(np.arange(ITEMS + 1), rows)
        for a, b in zip(before, after):
            assert torch.equal(_table(eng, a)[keep], _table(eng, b)[keep]), step
        for name, off in eng.offsets.items():
            if name.endswith("k.b"):    # analytically zero gradient: its Adam direction is the sign of rounding noise
                continue
            n = eng.P[name].numel()
            for dev_flat, host in ((after[0], p), (after[1], ref.m), (after[2], ref.v)):
                assert rel_err(dev_flat[off:off + n].numpy(), host[name].reshape(-1).numpy()) <= 1e-4, (step, name)
    for a, b in zip(w0, _state(eng)):
        assert torch.equal(_table(eng, a)[0], _table(eng, b)[0])


@pytest.mark.emu
def test_two_runs_are_bitwise_identical():
    runs = []
    for _ in range(2):
        eng = _engine("emu", "sasrec", "lazy_adam", dropout_rate=0.3)
        for step in range(3):
            eng.launch_train_step(_load(eng, _batch(step)))
        runs.append(_state(eng))
    for a, b in zip(*runs):
        assert torch.equal(a, b)


@pytest.mark.emu
def test_construction_rejects_l2_and_unknown_names():
    with pytest.raises(ValueError, match="l2_emb"):
        _engine("emu", "sasrec", "lazy_adam", l2_emb=1e-4)
    with pytest.raises(ValueError, match="optimizer"):
        _engine("emu", "sasrec", "sgd")
    assert _engine("emu", "sasrec", "adam", l2_emb=1e-4).stamp is None


@pytest.mark.emu
def test_backward_passes_without_adam_rewrite_the_touched_rows():
    """each backward pass gets a fresh epoch: a second pass with no optimizer step in between writes the touched rows
    again instead of adding to them, and they carry the dense path's bits"""
    gb = _batch(1)
    rows = _touched(gb)
    grads = []
    for opt, passes in (("adam", 1), ("lazy_adam", 1), ("lazy_adam", 2)):
        eng = _engine("emu", "sasrec", opt)
        c = _load(eng, gb)
        for _ in range(passes):
            eng.launch_fwd_bwd(c)
        grads.append(eng.G["item_emb"].cpu().clone()[rows])
    assert grads[0].abs().sum() > 0
    assert torch.equal(grads[0], grads[1]) and torch.equal(grads[0], grads[2])


# ---------------------------------------------------------------------------------------------------- world 2 (gloo)
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, shard, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    from cast_b200 import dist as cdist
    cdist.init_from_env("gloo")
    lib, dev = backend("emu")
    args = make_args(hidden_units=H, maxlen=T, num_heads=2, num_blocks=1, dropout_rate=0.0, optimizer="lazy_adam")
    arena = cdist.PeerArena(lib, dev) if shard else None
    eng = Engine("sasrec", 80, ITEMS, args, device=dev, lib=lib, seed=5 if shard else 5 + rank,
                 item_shard=(rank, world) if shard else None, alloc=arena.alloc if shard else None)
    cdist.attach(eng, arena=arena)
    per = B // world
    steps = 2
    for step in range(steps):
        eng.launch_train_step(_load(eng, _batch(step), rank * per, (rank + 1) * per))
    flat = [[torch.zeros_like(t) for _ in range(world)] for t in (eng.w, eng.m, eng.v)]
    for parts, t in zip(flat, (eng.w, eng.m, eng.v)):
        dist.all_gather(parts, t.clone())
    if rank == 0:
        single = Engine("sasrec", 80, ITEMS, args, device=dev, lib=lib, seed=5)
        init = single.w.clone()
        for step in range(steps):
            single.launch_train_step(_load(single, _batch(step)))
        torch.save({"parts": [[x.numpy().copy() for x in f] for f in flat], "init": init.numpy().copy(),
                    "single": [t.numpy().copy() for t in (single.w, single.m, single.v)],
                    "offsets": dict(single.offsets), "sizes": {k: v.numel() for k, v in single.P.items()},
                    "region": eng.P["item_emb"].numel(), "shard_R": eng.shard_R}, out)
    dist.barrier()
    if arena is not None:
        arena.close()
    dist.destroy_process_group()


def _unshard(flat_per_rank, R, V):
    full = np.zeros((V, H), np.float32)
    for q, flat in enumerate(flat_per_rank):
        sh = flat[:R * H].reshape(R, H)
        ids = np.arange(q, V, len(flat_per_rank))
        full[ids] = sh[(1 if q else 0):(1 if q else 0) + len(ids)]
    return full


@pytest.mark.emu
@pytest.mark.parametrize("shard", [False, True], ids=["replicated", "row_sharded"])
def test_two_ranks_equal_one_process(tmp_path, shard):
    """2 ranks with half the batch each against one process on the whole batch, 2 lazy steps.  Replicated: every rank's
    Adam sums the touching ranks' rows (each rank's stamps against its own epoch).  Row-sharded: the owner pull writes
    or adds by the owner's stamps.  Rows touched by only one rank exist in both steps."""
    out = str(tmp_path / "res.pt")
    mp.spawn(_worker, args=(2, _free_port(), shard, out), nprocs=2, join=True)
    r = torch.load(out, weights_only=False)
    V = ITEMS + 1
    n1 = r["sizes"]["item_emb"]
    for step in range(2):
        gb = _batch(step)
        one_rank = np.setxor1d(_touched(gb, 0, B // 2), _touched(gb, B // 2, B))
        assert len(one_rank) > 10
    touched = np.union1d(_touched(_batch(0)), _touched(_batch(1)))
    untouched = np.setdiff1d(np.arange(V), touched)
    init_tab = r["init"][:n1].reshape(V, H)
    for i, name in enumerate(("w", "m", "v")):
        single = r["single"][i]
        parts = r["parts"][i]
        tab1 = single[:n1].reshape(V, H)
        tab = _unshard(parts, r["shard_R"], V) if shard else parts[0][:n1].reshape(V, H)
        if not shard:
            assert np.array_equal(parts[0], parts[1])           # replicas identical
        assert np.array_equal(tab[untouched], tab1[untouched]), name
        if name == "w":
            assert np.array_equal(tab[untouched], init_tab[untouched])
            assert not np.array_equal(tab[touched], init_tab[touched])
            assert np.abs(tab - tab1).max() <= 2e-5
        else:
            assert rel_err(tab, tab1) <= (2e-5 if name == "m" else 4e-5), name
        region = r["region"]
        for k, off in r["offsets"].items():
            if k == "item_emb" or k.endswith("k.b"):
                continue
            n = r["sizes"][k]
            a = parts[0][region + off - n1: region + off - n1 + n]
            b = single[off:off + n]
            if name == "w":
                assert np.abs(a - b).max() <= 2e-5, (name, k)
            else:
                assert rel_err(a, b) <= (2e-5 if name == "m" else 4e-5), (name, k)
    if shard:
        for i in range(3):                                       # the pad row of rank 1 never moves
            assert not r["parts"][i][1][:H].any()


@pytest.mark.emu
def test_driver_trains_with_lazy_adam(tmp_path):
    import main as driver
    lib, dev = backend("emu")
    here = os.path.dirname(os.path.abspath(__file__))
    argv = ["--dataset", os.path.join(here, "golden", "ref_dataset.txt"), "--train_dir", "lazy", "--model", "sasrec",
            "--maxlen", "8", "--hidden_units", "12", "--batch_size", "16", "--num_epochs", "1", "--dropout_rate", "0.2",
            "--eval_every", "1", "--eval_batch", "40", "--model_path", str(tmp_path), "--optimizer", "lazy_adam"]
    assert driver.run(driver.build_parser().parse_args(argv), device=dev, lib=lib) == 0
    run_dir = os.path.join(str(tmp_path), "ref_dataset.txt")
    (sub,) = os.listdir(run_dir)
    assert json.load(open(os.path.join(run_dir, sub, "params.txt")))["optimizer"] == "lazy_adam"


# ---------------------------------------------------------------------------------------------------------- B200
def _gpu_model(use_graph, optimizer="lazy_adam"):
    import cast_b200
    args = make_args(hidden_units=50, maxlen=50, num_heads=1, num_blocks=2, dropout_rate=0.2, optimizer=optimizer)
    return cast_b200.SASRec(80, ITEMS, args, use_graph=use_graph, seed=11)


def _gpu_step(m, i):
    gb = golden_batch(tag="lin" if i % 2 == 0 else "log", idx=i % 3)
    return m.train_step(gb["u"], gb["seq"], gb["pos"], gb["neg"])


@pytest.mark.gpu
def test_gpu_graph_replay_equals_eager():
    """use_graph=True (with _capture's eager warm-up step and parameter restore) against eager launches: same bits"""
    a, b = _gpu_model(True), _gpu_model(False)
    for i in range(6):
        assert _gpu_step(a, i) == _gpu_step(b, i)
    for x, y in zip(_state(a.engine), _state(b.engine)):
        assert torch.equal(x, y)


@pytest.mark.gpu
def test_gpu_first_step_equals_dense_and_untouched_rows_stay():
    a, b = _gpu_model(False), _gpu_model(False, "adam")
    assert _gpu_step(a, 0) == _gpu_step(b, 0)
    for x, y in zip(_state(a.engine), _state(b.engine)):
        assert torch.equal(x, y)
    before = _state(a.engine)
    _gpu_step(a, 1)
    keep = np.setdiff1d(np.arange(ITEMS + 1), _touched(golden_batch(tag="log", idx=1)))
    assert len(keep) > 0
    for x, y in zip(before, _state(a.engine)):
        assert torch.equal(_table(a.engine, x)[keep], _table(a.engine, y)[keep])


@pytest.mark.gpu
def test_gpu_checkpoint_resume_is_bit_identical(tmp_path):
    from cast_b200 import checkpoint as ck
    a = _gpu_model(True)
    for i in range(3):
        _gpu_step(a, i)
    prefix = ck.save_model(str(tmp_path / "model.ckpt"), a, "sasrec", 2)
    b = _gpu_model(True)
    ck.restore_model(prefix, b, "sasrec", 2)
    for i in range(3, 6):
        assert _gpu_step(a, i) == _gpu_step(b, i)
    for x, y in zip(_state(a.engine), _state(b.engine)):
        assert torch.equal(x, y)


@pytest.mark.gpu
def test_gpu_driver_trains_with_lazy_adam(tmp_path):
    import main as driver
    here = os.path.dirname(os.path.abspath(__file__))
    argv = ["--dataset", os.path.join(here, "golden", "ref_dataset.txt"), "--train_dir", "lazy", "--model", "sasrec",
            "--maxlen", "50", "--batch_size", "32", "--num_epochs", "1", "--eval_every", "1",
            "--model_path", str(tmp_path), "--optimizer", "lazy_adam"]
    assert driver.run(driver.build_parser().parse_args(argv)) == 0
    run_dir = os.path.join(str(tmp_path), "ref_dataset.txt")
    (sub,) = os.listdir(run_dir)
    assert json.load(open(os.path.join(run_dir, sub, "params.txt")))["optimizer"] == "lazy_adam"
