"""Global-norm gradient clipping (args.clip_grad with threshold args.max_norm, tf.clip_by_global_norm over the gradient
Adam consumes), computed on the device inside the step.  A step below the threshold gives the bits of clipping off; a
clipped step tracks the oracle's gradients through clip_by_global_norm (float64, below) + TF-Adam; data-parallel runs
(replicated and row-sharded) agree with one process.  Host-emulated kernels (`emu`, CPU) at tiny shapes and the B200
(`gpu`)."""
import logging
import math
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from helpers import (O, backend, dropout_hook, golden_batch, make_args, oracle_batch, rel_err, relu_kink_hook,
                     synth_batch)
from cast_b200.engine import Engine

B, T, H = 4, 10, 12
ITEMS = 300


def _args(optimizer="adam", **kw):
    return make_args(**{"hidden_units": H, "maxlen": T, "num_heads": 2, "num_blocks": 1, "dropout_rate": 0.0,
                        "optimizer": optimizer, **kw})


def _engine(model, optimizer="adam", seed=5, **kw):
    lib, dev = backend("emu")
    return Engine(model, 80, ITEMS, _args(optimizer, **kw), device=dev, lib=lib, seed=seed)


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


def clip_by_global_norm(grads, max_norm):
    """tf.clip_by_global_norm in float64: norm = sqrt(sum of every gradient's squares); every gradient is multiplied by
    max_norm / norm if norm > max_norm (NaN for a non-finite norm).  Returns (clipped float64 grads, norm)."""
    norm = math.sqrt(sum(float((g.double() ** 2).sum()) for g in grads.values()))
    if not math.isfinite(norm):
        scale = float("nan")
    else:
        scale = max_norm / norm if norm > max_norm else 1.0
    return {k: g.double() * scale for k, g in grads.items()}, norm


def _state(eng):
    return eng.w.cpu().clone(), eng.m.cpu().clone(), eng.v.cpu().clone(), eng.adam_state.cpu().clone()


class _ClippedTFAdam(O.TFAdam):
    """float64 reference: TF-Adam on the given (clipped) gradients; with `rows`, the item table is updated on those rows
    only (LazyAdam)"""

    def step(self, params, grads, rows=None):
        lr_t = np.float64(np.float32(self.lr) * np.sqrt(np.float32(1) - self.b2p) / (np.float32(1) - self.b1p))
        with torch.no_grad():
            for k, w in params.items():
                sel = torch.from_numpy(rows) if (k == "item_emb" and rows is not None) else slice(None)
                g, m, v = grads[k][sel], self.m[k][sel], self.v[k][sel]
                m = self.b1 * m + (1 - self.b1) * g
                v = self.b2 * v + (1 - self.b2) * g * g
                w[sel] = w[sel] - lr_t * m / (v.sqrt() + self.eps)
                self.m[k][sel], self.v[k][sel] = m, v
        self.b1p = np.float32(self.b1p * np.float32(self.b1))
        self.b2p = np.float32(self.b2p * np.float32(self.b2))


def _randomize_beta(eng):
    # beta != 0: with beta = 0 the reference's query mask sign(|sum_H LN(x)|) is decided by rounding noise (DESIGN.md)
    g = torch.Generator().manual_seed(3)
    eng.load_parameters({k: torch.randn(v.shape, generator=g) * 0.1 for k, v in eng.P.items() if k.endswith("beta")})


def _first_norm(model, args, eng):
    p = {k: v.detach().cpu().float().clone() for k, v in eng.P.items()}
    _, _, grads = O.train_step(model, p, None, args, oracle_batch(_batch(0)))
    return clip_by_global_norm(grads, 1.0)[1]


@pytest.mark.emu
@pytest.mark.parametrize("optimizer", ["adam", "lazy_adam"])
@pytest.mark.parametrize("model", ["sasrec", "cast_4"])
def test_large_threshold_is_bit_identical_to_clipping_off(model, optimizer):
    out = []
    for kw in ({}, {"clip_grad": True, "max_norm": 1e30}):
        eng = _engine(model, optimizer, **kw)
        for step in range(3):
            eng.launch_train_step(_load(eng, _batch(step)))
        out.append(_state(eng))
    for a, b in zip(*out):
        assert torch.equal(a, b)


@pytest.mark.emu
@pytest.mark.parametrize("model,optimizer,l2", [("sasrec", "adam", 0.0), ("sasrec", "adam", 1e-3),
                                                ("cast_4", "adam", 0.0), ("sasrec", "lazy_adam", 0.0),
                                                ("cast_4", "lazy_adam", 0.0)])
def test_clipped_steps_track_reference(model, optimizer, l2):
    """4 steps on reference-sampler batches with max_norm = 0.25 x the oracle's first-step norm: every step clips, the
    device norm matches the oracle's within 1e-5 relative, and w, m, v match clip_by_global_norm + (lazy) TF-Adam in
    float64 within 1e-4 relative"""
    probe = _engine(model, optimizer, l2_emb=l2)
    _randomize_beta(probe)
    max_norm = 0.25 * _first_norm(model, probe.args, probe)
    eng = _engine(model, optimizer, l2_emb=l2, clip_grad=True, max_norm=max_norm)
    _randomize_beta(eng)
    args = eng.args
    p = {k: v.detach().cpu().double().clone() for k, v in eng.P.items()}
    ref = _ClippedTFAdam(p, lr=args.lr)
    for step in range(4):
        gb = _batch(step)
        eng.launch_train_step(_load(eng, gb))
        _, _, grads = O.train_step(model, {k: v.float() for k, v in p.items()}, None, args, oracle_batch(gb))
        clipped, norm_o = clip_by_global_norm(grads, max_norm)
        scale, norm = eng.clip_out.cpu().tolist()
        assert norm > max_norm and scale < 1.0, step
        assert abs(norm - norm_o) <= 1e-5 * norm_o, (step, norm, norm_o)
        ref.step(p, clipped, _touched(gb) if optimizer == "lazy_adam" else None)
        for name, off in eng.offsets.items():
            if name.endswith("k.b"):    # analytically zero gradient: its Adam direction is the sign of rounding noise
                continue
            n = eng.P[name].numel()
            for dev_flat, host in ((eng.w, p), (eng.m, ref.m), (eng.v, ref.v)):
                assert rel_err(dev_flat[off:off + n].numpy(), host[name].reshape(-1).numpy()) <= 1e-4, (step, name)


@pytest.mark.emu
@pytest.mark.parametrize("optimizer", ["adam", "lazy_adam"])
def test_two_clipped_runs_are_bitwise_identical(optimizer):
    runs = []
    for _ in range(2):
        eng = _engine("sasrec", optimizer, dropout_rate=0.3, clip_grad=True, max_norm=0.05)
        norms = []
        for step in range(3):
            eng.launch_train_step(_load(eng, _batch(step)))
            norms.append(eng.clip_out.clone())
        assert all(float(x[1]) > 0.05 for x in norms)
        runs.append(_state(eng) + tuple(norms))
    for a, b in zip(*runs):
        assert torch.equal(a, b)


@pytest.mark.emu
def test_construction_errors_and_off_state():
    import cast_b200
    for bad in (0.0, -1.0, float("inf"), float("nan")):
        with pytest.raises(ValueError, match="max_norm"):
            _engine("sasrec", clip_grad=True, max_norm=bad)
    assert _engine("sasrec", max_norm=-1.0).clip_out is None      # the threshold is unused without clip_grad
    lib, dev = backend("emu")
    m = cast_b200.SASRec(80, ITEMS, _args(), device=dev, _lib=lib, use_graph=False)
    gb = _batch(0)
    m.train_step(gb["u"], gb["seq"], gb["pos"], gb["neg"])
    assert m.last_grad_norm() is None
    m = cast_b200.SASRec(80, ITEMS, _args(clip_grad=True, max_norm=1e30), device=dev, _lib=lib, use_graph=False)
    m.train_step(gb["u"], gb["seq"], gb["pos"], gb["neg"])
    assert m.last_grad_norm() == float(m.engine.clip_out[1]) > 0


# ---------------------------------------------------------------------------------------------------- world 2 (gloo)
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


MAX_NORM_DP = 0.05     # below every step's norm at these shapes (asserted)


def _worker(rank, world, port, shard, optimizer, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    from cast_b200 import dist as cdist
    cdist.init_from_env("gloo")
    lib, dev = backend("emu")
    args = _args(optimizer, clip_grad=True, max_norm=MAX_NORM_DP)
    arena = cdist.PeerArena(lib, dev) if shard else None
    eng = Engine("sasrec", 80, ITEMS, args, device=dev, lib=lib, seed=5 if shard else 5 + rank,
                 item_shard=(rank, world) if shard else None, alloc=arena.alloc if shard else None)
    cdist.attach(eng, arena=arena)
    per = B // world
    steps = 2
    norms = []
    for step in range(steps):
        eng.launch_train_step(_load(eng, _batch(step), rank * per, (rank + 1) * per))
        norms.append(eng.clip_out.clone())
    flat = [[torch.zeros_like(t) for _ in range(world)] for t in (eng.w, eng.m, eng.v)]
    for parts, t in zip(flat, (eng.w, eng.m, eng.v)):
        dist.all_gather(parts, t.clone())
    all_norms = [torch.zeros(steps, 2) for _ in range(world)]
    dist.all_gather(all_norms, torch.stack(norms))
    if rank == 0:
        single = Engine("sasrec", 80, ITEMS, args, device=dev, lib=lib, seed=5)
        single_norms = []
        for step in range(steps):
            single.launch_train_step(_load(single, _batch(step)))
            single_norms.append(single.clip_out.clone())
        torch.save({"parts": [[x.numpy().copy() for x in f] for f in flat],
                    "norms": [x.numpy().copy() for x in all_norms],
                    "single_norms": torch.stack(single_norms).numpy(),
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


def _check_two_ranks(r, shard):
    V = ITEMS + 1
    n1 = r["sizes"]["item_emb"]
    norms = r["norms"]
    assert np.array_equal(norms[0], norms[1])                    # every rank folds the same values in the same order
    assert (norms[0][:, 1] > MAX_NORM_DP).all() and (norms[0][:, 0] < 1).all()
    assert np.abs(norms[0][:, 1] - r["single_norms"][:, 1]).max() <= 1e-5 * r["single_norms"][:, 1].max()
    for i, name in enumerate(("w", "m", "v")):
        single, parts = r["single"][i], r["parts"][i]
        if not shard:
            assert np.array_equal(parts[0], parts[1])           # replicas identical
        tab = _unshard(parts, r["shard_R"], V) if shard else parts[0][:n1].reshape(V, H)
        tab1 = single[:n1].reshape(V, H)
        assert np.abs(tab - tab1).max() <= 1e-5 * np.abs(tab1).max(), name
        region = r["region"]
        for k, off in r["offsets"].items():
            if k == "item_emb" or k.endswith("k.b"):
                continue
            n = r["sizes"][k]
            a = parts[0][region + off - n1: region + off - n1 + n]
            b = single[off:off + n]
            assert np.abs(a - b).max() <= 1e-5 * max(np.abs(b).max(), 1e-30), (name, k)


@pytest.mark.emu
@pytest.mark.parametrize("optimizer", ["adam", "lazy_adam"])
@pytest.mark.parametrize("shard", [False, True], ids=["replicated", "row_sharded"])
def test_two_ranks_equal_one_process(tmp_path, shard, optimizer):
    """2 ranks with half the batch each against one process on the whole batch, 2 clipped steps: replicas bit-identical,
    the same norm bits on every rank, every tensor within 1e-5 of its largest magnitude"""
    out = str(tmp_path / "res.pt")
    mp.spawn(_worker, args=(2, _free_port(), shard, optimizer, out), nprocs=2, join=True)
    _check_two_ranks(torch.load(out, weights_only=False), shard)


@pytest.mark.emu
def test_driver_logs_grad_norm(tmp_path):
    import main as driver
    lib, dev = backend("emu")
    here = os.path.dirname(os.path.abspath(__file__))
    argv = ["--dataset", os.path.join(here, "golden", "ref_dataset.txt"), "--train_dir", "clip", "--model", "sasrec",
            "--maxlen", "8", "--hidden_units", "12", "--batch_size", "16", "--num_epochs", "1", "--dropout_rate", "0.2",
            "--eval_every", "1", "--eval_batch", "40", "--model_path", str(tmp_path), "--clip_grad", "--max_norm", "1.0"]
    lines = []

    class _Keep(logging.Handler):
        def emit(self, record):
            lines.append(record.getMessage())

    logger = logging.getLogger("grad_clip_driver")
    logger.setLevel(logging.INFO)
    logger.addHandler(_Keep())
    assert driver.run(driver.build_parser().parse_args(argv), device=dev, lib=lib, logger=logger) == 0
    epoch = [ln for ln in lines if "TRAIN/loss" in ln]
    assert len(epoch) == 1 and "TRAIN/grad_norm" in epoch[0]
    assert float(epoch[0].split("TRAIN/grad_norm")[1]) > 0


# ---------------------------------------------------------------------------------------------------------- B200
ADDED_LAUNCHES = {"adam": 2, "lazy_adam": 3}    # single process (DESIGN.md §7b lists every path)


def _gpu_reference_step(eng, p_dev, grads, max_norm, rows, lr):
    """clip_by_global_norm + (lazy) TF-Adam in float64 from the device's own state before the step"""
    w0, m0, v0, st = p_dev
    clipped, norm = clip_by_global_norm(grads, max_norm)
    b1p, b2p = st
    lr_t = float(np.float32(lr) * np.sqrt(np.float32(1) - b2p) / (np.float32(1) - b1p))
    ref = {}
    for k, off in eng.offsets.items():
        n = eng.P[k].numel()
        g = clipped[k].reshape(-1)
        w, m, v = (t[off:off + n].double().clone() for t in (w0, m0, v0))
        sel = slice(None)
        if k == "item_emb" and rows is not None:
            sel = torch.from_numpy((rows[:, None] * eng.H + np.arange(eng.H)[None, :]).reshape(-1))
        m[sel] = 0.9 * m[sel] + 0.1 * g[sel]
        v[sel] = 0.98 * v[sel] + 0.02 * g[sel] * g[sel]
        w[sel] = w[sel] - lr_t * m[sel] / (v[sel].sqrt() + 1e-8)
        ref[k] = (w, m, v)
    return ref, norm


@pytest.mark.gpu
@pytest.mark.parametrize("optimizer", ["adam", "lazy_adam"])
@pytest.mark.parametrize("shape", ["c2", "wide"])
def test_gpu_clipped_steps_match_oracle(shape, optimizer):
    """C2 (B 128, T 200, H 50) and a wide table (H 256, 50 000 items), 2 clipped steps: each step against the oracle's
    gradients at the device's own parameters (ReLU kinks resolved as the device resolved them), clipped in float64,
    then TF-Adam from the device's state before the step"""
    lib, dev = backend("gpu")
    Bs, Ts, Hs, items, heads = (128, 200, 50, 300, 1) if shape == "c2" else (32, 50, 256, 50000, 2)
    rate = 0.2
    args = make_args(hidden_units=Hs, maxlen=Ts, num_heads=heads, num_blocks=2, dropout_rate=rate,
                     optimizer=optimizer, clip_grad=True)
    probe = Engine("sasrec", 80, items, args, device=dev, lib=lib, seed=7)
    gb0 = synth_batch(Bs, Ts, items, seed=0)
    p = {k: v.detach().cpu().clone() for k, v in probe.P.items()}
    _, _, g0 = O.train_step("sasrec", p, None, args, oracle_batch(gb0))
    args.max_norm = 0.25 * clip_by_global_norm(g0, 1.0)[1]
    eng = Engine("sasrec", 80, items, args, device=dev, lib=lib, seed=7)
    _randomize_beta(eng)
    for step in range(2):
        gb = synth_batch(Bs, Ts, items, seed=step)
        c = eng.ctx(Bs)
        c.keys3.copy_(torch.from_numpy(np.stack([gb[k].reshape(-1) for k in ("seq", "pos", "neg")])))
        before = (eng.w.cpu().clone(), eng.m.cpu().clone(), eng.v.cpu().clone(),
                  eng.adam_state[:1].cpu().view(torch.float32).numpy().copy())
        p = {k: v.detach().cpu().clone() for k, v in eng.P.items()}
        eng.launch_fwd_bwd(c)
        with relu_kink_hook(eng, c, rate) as kink:
            _, _, grads = O.train_step("sasrec", p, None, args, oracle_batch(gb), dropout_hook(eng, rate))
        assert kink.ambiguous <= max(8, 2e-4 * kink.total), (kink.ambiguous, kink.total)
        eng.adam(c)
        rows = _touched(gb) if optimizer == "lazy_adam" else None
        ref, norm_o = _gpu_reference_step(eng, before, grads, args.max_norm, rows, args.lr)
        scale, norm = eng.clip_out.cpu().tolist()
        assert norm > args.max_norm and scale < 1.0
        assert abs(norm - norm_o) <= 1e-4 * norm_o, (step, norm, norm_o)
        for k, off in eng.offsets.items():
            if k.endswith("k.b"):
                continue
            n = eng.P[k].numel()
            w, m, v = ref[k]
            assert rel_err(eng.m[off:off + n].cpu().numpy(), m.numpy()) <= 1e-4, (step, k, "m")
            assert rel_err(eng.v[off:off + n].cpu().numpy(), v.numpy()) <= 2e-4, (step, k, "v")
            # elements whose gradient sits at the rounding floor move by a fraction of lr either way (smoke())
            assert rel_err(eng.w[off:off + n].cpu().numpy(), w.numpy()) <= 3e-4, (step, k, "w")


def _gpu_model(use_graph, optimizer, **kw):
    import cast_b200
    args = make_args(hidden_units=50, maxlen=50, num_heads=1, num_blocks=2, dropout_rate=0.2, optimizer=optimizer,
                     **kw)
    return cast_b200.SASRec(80, ITEMS, args, use_graph=use_graph, seed=11)


def _gpu_step(m, i):
    gb = golden_batch(tag="lin" if i % 2 == 0 else "log", idx=i % 3)
    return m.train_step(gb["u"], gb["seq"], gb["pos"], gb["neg"])


@pytest.mark.gpu
@pytest.mark.parametrize("optimizer", ["adam", "lazy_adam"])
def test_gpu_graph_replay_equals_eager_with_clipping(optimizer):
    a = _gpu_model(True, optimizer, clip_grad=True, max_norm=0.05)
    b = _gpu_model(False, optimizer, clip_grad=True, max_norm=0.05)
    for i in range(6):
        assert _gpu_step(a, i) == _gpu_step(b, i)
        na, nb = a.last_grad_norm(), b.last_grad_norm()
        assert na == nb and na > 0.05
    for x, y in zip(_state(a.engine), _state(b.engine)):
        assert torch.equal(x, y)


@pytest.mark.gpu
@pytest.mark.parametrize("optimizer", ["adam", "lazy_adam"])
def test_gpu_large_threshold_equals_clipping_off_and_launch_counts(optimizer):
    """graph replay with max_norm = 1e30 gives the bits of clipping off; the captured step issues the launches of a
    model built without the option, plus ADDED_LAUNCHES with clipping on"""
    plain = _gpu_model(True, optimizer)
    off = _gpu_model(True, optimizer, clip_grad=False)
    on = _gpu_model(True, optimizer, clip_grad=True, max_norm=1e30)
    for i in range(4):
        r = _gpu_step(plain, i)
        assert _gpu_step(off, i) == r and _gpu_step(on, i) == r
    for x, y, z in zip(_state(plain.engine), _state(off.engine), _state(on.engine)):
        assert torch.equal(x, y) and torch.equal(x, z)
    assert off.launches_per_step == plain.launches_per_step
    assert on.launches_per_step == plain.launches_per_step + ADDED_LAUNCHES[optimizer]


# ------------------------------------------------------------------------------------------------------ 2 x B200
def _gpu_worker(rank, world, port, shard, optimizer, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    from cast_b200 import dist as cdist
    cdist.init_from_env("nccl")
    lib, dev = backend("gpu")
    dev = torch.device("cuda", rank)
    args = _args(optimizer, clip_grad=True, max_norm=MAX_NORM_DP)
    eng = Engine("sasrec", 80, ITEMS, args, device=dev, lib=lib, seed=5 if shard else 5 + rank,
                 item_shard=(rank, world) if shard else None)
    cdist.attach(eng)
    per = B // world
    norms = []
    for step in range(2):
        eng.launch_train_step(_load(eng, _batch(step), rank * per, (rank + 1) * per))
        norms.append(eng.clip_out.clone())
    torch.cuda.synchronize(dev)
    flat = [[torch.zeros_like(t) for _ in range(world)] for t in (eng.w, eng.m, eng.v)]
    for parts, t in zip(flat, (eng.w, eng.m, eng.v)):
        dist.all_gather(parts, t.clone())
    all_norms = [torch.zeros(2, 2, device=dev) for _ in range(world)]
    dist.all_gather(all_norms, torch.stack(norms))
    if rank == 0:
        single = Engine("sasrec", 80, ITEMS, args, device=dev, lib=lib, seed=5)
        single_norms = []
        for step in range(2):
            single.launch_train_step(_load(single, _batch(step)))
            single_norms.append(single.clip_out.clone())
        torch.save({"parts": [[x.cpu().numpy().copy() for x in f] for f in flat],
                    "norms": [x.cpu().numpy().copy() for x in all_norms],
                    "single_norms": torch.stack(single_norms).cpu().numpy(),
                    "single": [t.cpu().numpy().copy() for t in (single.w, single.m, single.v)],
                    "offsets": dict(single.offsets), "sizes": {k: v.numel() for k, v in single.P.items()},
                    "region": eng.P["item_emb"].numel(), "shard_R": eng.shard_R}, out)
    cdist.quiesce(eng)
    if eng.arena is not None:
        eng.arena.close()
    dist.destroy_process_group()


@pytest.mark.gpu
@pytest.mark.parametrize("optimizer", ["adam", "lazy_adam"])
@pytest.mark.parametrize("shard", [False, True], ids=["replicated", "row_sharded"])
def test_gpu_two_ranks_equal_one_process(tmp_path, shard, optimizer):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two visible GPUs")
    out = str(tmp_path / "res.pt")
    mp.spawn(_gpu_worker, args=(2, _free_port(), shard, optimizer, out), nprocs=2, join=True)
    _check_two_ranks(torch.load(out, weights_only=False), shard)
