"""End-to-end parity of one training step and of evaluation scoring: kernels (through the C ABI and the model
classes) vs the CPU oracle on batches produced by the REFERENCE's own sampler (tests/golden/ref_sampler.npz).

Tolerance (BASELINE.json north_star): fp32 within 1e-4 relative for logits / loss; gradients are compared per
tensor relative to that tensor's max magnitude.  The key-projection bias gradient is analytically zero (a constant
added to every key shifts all scores of a softmax row equally) so it is compared absolutely against the scale of
the query-bias gradient.  ReLU kinks: a hidden unit whose pre-activation is within 2e-5 of zero has an
implementation-defined derivative (its sign is fp32 noise); for those units — a handful per block — the oracle takes
the device's decision (helpers.relu_kink_hook, count asserted negligible), everywhere else its own.  Runs on the GPU (`-m gpu`, real library) and, at tiny shapes, on the host-emulated
kernel sources (`emu`, CPU, test infrastructure only).
"""
import numpy as np
import pytest
import torch

from helpers import O, backend, dropout_hook, golden_batch, make_args, oracle_batch, rel_err, relu_kink_hook
from cast_b200.engine import Engine

TOL = 1e-4


def run_step(kind, model, B, T, H, heads, rate, seed=7, randomize=True, blocks=2, tag="lin", l2=0.0, gb=None,
             itemnum=300):
    lib, dev = backend(kind)
    args = make_args(hidden_units=H, maxlen=T, num_heads=heads, num_blocks=blocks, dropout_rate=rate, l2_emb=l2)
    if gb is None:
        gb = golden_batch(tag=tag, B=B, T=T)
    eng = Engine(model, 80, itemnum, args, device=dev, lib=lib, seed=seed)
    p = {k: v.detach().cpu().clone() for k, v in eng.P.items()}
    if randomize:  # non-trivial beta/gamma/biases so that query masks, residual LN paths etc. are exercised
        g = torch.Generator().manual_seed(3)
        for k in p:
            if k.endswith(".b") or k.endswith("beta"):
                p[k] = torch.randn(p[k].shape, generator=g) * 0.1
            if k.endswith("gamma"):
                p[k] = 1 + torch.randn(p[k].shape, generator=g) * 0.1
        eng.load_parameters(p)
    c = eng.ctx(B)
    c.keys3.copy_(torch.from_numpy(np.stack([gb[k].reshape(-1) for k in ("seq", "pos", "neg")])))
    c.cids.copy_(torch.from_numpy(np.stack([gb[k].reshape(-1) for k in ("timeseq", "hours", "days")])))
    opt = O.TFAdam(p, lr=args.lr)
    # device forward + backward first (the step counter, hence the dropout masks, stays put until Adam runs), then the
    # oracle with the identical dropout masks and the ReLU kinks resolved as the device resolved them, then Adam
    eng.launch_fwd_bwd(c)
    with relu_kink_hook(eng, c, rate) as kink:
        auc_o, loss_o, grads_o = O.train_step(model, p, opt, args, oracle_batch(gb), dropout_hook(eng, rate))
    assert kink.ambiguous <= max(8, 2e-4 * kink.total), (kink.ambiguous, kink.total)
    if eng.grad_allreduce is not None:
        eng.grad_allreduce(c)
    eng.adam(c)
    if eng.after_adam is not None:
        eng.after_adam()
    s = eng.sums[:3].tolist()
    return eng, p, grads_o, (auc_o, loss_o), s


def check_step(eng, p, grads_o, ref, s, tol=TOL):
    auc_o, loss_o = ref
    loss, auc, cnt = s[0] / s[2], s[1] / s[2], s[2]
    assert abs(loss - loss_o) <= tol * abs(loss_o)
    assert abs(auc - auc_o) <= 1e-6
    for k in eng.G:
        go = grads_o[k].numpy().astype(np.float64) * cnt  # engine gradients are un-normalised
        gk = eng.G[k].cpu().numpy()
        if k.endswith("k.b"):
            scale = np.abs(grads_o[k.replace("k.b", "q.b")].numpy()).max() * cnt
            assert np.abs(gk - go).max() <= 1e-4 * max(scale, 1e-20), k
        else:
            assert rel_err(gk, go) <= tol, (k, rel_err(gk, go))
    assert eng.state_step() == 1


EMU_CASES = [("sasrec", 3, 12, 20, 2, 0.25), ("sasrec_static", 7, 11, 12, 1, 0.2), ("cast_1", 2, 10, 12, 1, 0.3), ("cast_4", 2, 10, 12, 2, 0.2),
             ("cast_6", 2, 8, 12, 1, 0.2), ("cast_9", 2, 8, 8, 2, 0.1), ("sasrec", 2, 9, 40, 2, 0.2)]


@pytest.mark.emu
@pytest.mark.parametrize("model,B,T,H,heads,rate", EMU_CASES)
def test_train_step_emulated(model, B, T, H, heads, rate):
    check_step(*run_step("emu", model, B, T, H, heads, rate))


GPU_CASES = [(m, 16, 50, 50, 1, 0.2) for m in O.MODELS] + [
    ("sasrec", 16, 50, 50, 1, 0.0), ("sasrec", 8, 37, 50, 2, 0.5), ("cast_1", 16, 50, 50, 2, 0.2),
    ("sasrec", 4, 50, 128, 4, 0.2), ("sasrec", 4, 50, 256, 1, 0.2), ("cast_4", 8, 50, 64, 2, 0.3),
    ("sasrec", 8, 50, 100, 1, 0.1)]


@pytest.mark.gpu
@pytest.mark.parametrize("model,B,T,H,heads,rate", GPU_CASES)
def test_train_step_gpu(model, B, T, H, heads, rate):
    check_step(*run_step("gpu", model, B, T, H, heads, rate))


@pytest.mark.gpu
def test_train_step_gpu_logscale_batch():
    check_step(*run_step("gpu", "cast_3", 16, 50, 50, 1, 0.2, tag="log"))


@pytest.mark.gpu
def test_fused_and_unfused_paths_agree_at_full_size():
    """B=128, T=200 (400 row tiles: exercises the persistent backward loops): fused row kernels vs the generic GEMM
    path, same inputs -> gradients within 2e-5 relative (different summation order only)."""
    lib, dev = backend("gpu")
    args = make_args(hidden_units=50, maxlen=200, num_heads=1, num_blocks=2, dropout_rate=0.2)
    rng = np.random.RandomState(0)
    B, T = 128, 200
    seq = rng.randint(1, 301, (B, T)).astype(np.int32)
    lens = rng.randint(5, T + 1, B)
    for b in range(B):
        seq[b, :T - lens[b]] = 0
    pos = np.where(seq > 0, rng.randint(1, 301, (B, T)), 0).astype(np.int32)
    neg = np.where(seq > 0, rng.randint(1, 301, (B, T)), 0).astype(np.int32)
    outs = []
    for fused in (True, False):
        eng = Engine("sasrec", 80, 300, args, device=dev, lib=lib, seed=3, fused=fused)
        g = torch.Generator().manual_seed(5)
        for k in eng.P:
            if k.endswith("beta") or k.endswith(".b"):
                eng.P[k].copy_((torch.randn(eng.P[k].shape, generator=g) * 0.1).to(dev))
        c = eng.ctx(B)
        c.keys3.copy_(torch.from_numpy(np.stack([seq.reshape(-1), pos.reshape(-1), neg.reshape(-1)])))
        eng.launch_train_step(c)
        outs.append((eng.gbuf.cpu().numpy().copy(), eng.w.cpu().numpy().copy(), eng))
    ga, gb_ = outs[0][0], outs[1][0]
    assert abs(ga[-4] - gb_[-4]) <= 1e-5 * abs(gb_[-4])  # loss sum
    eng = outs[0][2]
    for k, off in eng.offsets.items():
        n = eng.P[k].numel()
        a, b = ga[off:off + n], gb_[off:off + n]
        if k.endswith("k.b"):
            continue
        assert rel_err(a, b) <= 2e-5, (k, rel_err(a, b))


@pytest.mark.gpu
def test_run_to_run_bitwise_determinism():
    """Same seed, same batch, two engines: every gradient bit-identical (no float atomics anywhere)."""
    a = run_step("gpu", "cast_1", 16, 50, 50, 2, 0.2)[0]
    b = run_step("gpu", "cast_1", 16, 50, 50, 2, 0.2)[0]
    assert torch.equal(a.gbuf, b.gbuf)
    assert torch.equal(a.w, b.w)


@pytest.mark.gpu
def test_multi_step_training_tracks_oracle():
    """5 consecutive steps on 3 different reference-sampler batches: loss trajectory within 1e-4 relative."""
    import cast_b200
    args = make_args(hidden_units=50, maxlen=50, num_heads=1, num_blocks=2, dropout_rate=0.2)
    model = cast_b200.SASRec(80, 300, args, use_graph=True)
    eng = model.engine
    p = {k: v.detach().cpu().clone() for k, v in eng.P.items()}
    # beta != 0: with the default init (gamma=1, beta=0) sum_H(LN(x)) is zero up to rounding, so the reference's
    # query mask sign(|sum_H queries|) (modules.py:248) is decided by rounding noise — see DESIGN.md "query-mask"
    g = torch.Generator().manual_seed(11)
    for k in p:
        if k.endswith("beta"):
            p[k] = torch.randn(p[k].shape, generator=g) * 0.1
    eng.load_parameters(p)
    opt = O.TFAdam(p, lr=args.lr)
    for step in range(5):
        gb = golden_batch(idx=step % 3)
        auc_o, loss_o, _ = O.train_step("sasrec", p, opt, args, oracle_batch(gb), dropout_hook(eng, 0.2))
        auc, loss = model.train_step(gb["u"], gb["seq"], gb["pos"], gb["neg"])
        assert abs(loss - loss_o) <= 2e-4 * abs(loss_o), (step, loss, loss_o)
    assert eng.state_step() == 5


@pytest.mark.gpu
def test_train_step_without_waiting_returns_the_previous_steps_metrics():
    """train_step(sync=False): same training (bit-equal weights), every step's (auc, loss) still read — one call later."""
    import cast_b200
    args = make_args(hidden_units=50, maxlen=50, num_heads=1, num_blocks=2, dropout_rate=0.2)
    a = cast_b200.SASRec(80, 300, args, use_graph=True)
    b = cast_b200.SASRec(80, 300, args, use_graph=True)
    b.engine.load_parameters({k: v.detach().cpu().clone() for k, v in a.engine.P.items()})
    waited, lagged = [], []
    for step in range(6):
        gb = golden_batch(idx=step % 3)
        waited.append(a.train_step(gb["u"], gb["seq"], gb["pos"], gb["neg"]))
        lagged.append(b.train_step(gb["u"], gb["seq"], gb["pos"], gb["neg"], sync=False))
    assert lagged[0] is None
    assert lagged[1:] == waited[:-1]
    assert b.last_metrics() == waited[-1]
    assert torch.equal(a.engine.w, b.engine.w)


@pytest.mark.gpu
@pytest.mark.parametrize("model", ["sasrec", "cast_1", "cast_7"])
def test_predict_matches_oracle(model):
    """models/sasrec.py:127-129 protocol: test_logits [B,101] within 1e-4, attention_weights [h*B,T,T] within 1e-5."""
    import cast_b200
    args = make_args(hidden_units=50, maxlen=50, num_heads=2, num_blocks=2, dropout_rate=0.2)
    m = cast_b200.build_model(model, 80, 300, 5, args)
    eng = m.engine
    p = {k: v.detach().cpu().clone() for k, v in eng.P.items()}
    g = torch.Generator().manual_seed(5)
    for k in p:  # trained-looking LN betas: padded query rows become live (SURVEY A-8)
        if k.endswith("beta"):
            p[k] = torch.randn(p[k].shape, generator=g) * 0.2
    eng.load_parameters(p)
    gb = golden_batch(B=4)
    item_idx = np.concatenate([[gb["pos"][0, -1]], np.random.RandomState(1).randint(1, 301, 100)]).astype(np.int32)
    logits, attn = m.predict(None, gb["u"], gb["seq"], item_idx, timeseq=gb["timeseq"], hours_seq=gb["hours"],
                             days_seq=gb["days"])
    seq, table, attn_o = O.forward(model, p, args, oracle_batch(gb))
    lo = O.test_logits(seq, table, item_idx).detach().numpy()
    assert logits.shape == (4, 101)
    assert rel_err(logits, lo) <= TOL
    assert attn.shape == tuple(attn_o.shape)
    assert np.abs(attn - attn_o.detach().numpy()).max() <= 1e-5
