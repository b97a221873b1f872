"""The block backward row kernels `cast_ffn_bwd`, `cast_qkv_bwd` and `cast_qkv_bwd_embed` (csrc/fused.cu,
csrc/fused_mma.cuh) against float64 torch autograd of the forward each one inverts (include/cast_b200.h):

  ffn:   zn = LN(y), h1d = relu(zn W1 + b1) * keep_h / (1 - r),
         xout = ((h1d W2 + b2) * keep_o / (1 - r) + zn) * (ids != 0), backpropagated with a given upstream gradient dx;
  qkv:   qn = LN(x), Q = qn Wq + bq, K = x Wk + bk, V = x Wv + bv, with random dQ, dK, dV and the attention residual's
         gradient dres added to d(qn);
  embed: the qkv gradient dx further multiplied by (ids != 0) * keep / (1 - r) at flat index row * H + col.

The saved activations the kernels read (zn, h1d, y, x, qn, mean, rstd) come from the float64 forward rounded to fp32,
so the ReLU / dropout activity the ffn kernel derives from `h1d > 0` is the reference's own; keep masks come from
`cast_dropout_keep` of the library under test.  Every parameter gradient is checked through the flat layout
`[ln.beta | ln.gamma | W | b | ...]` (k.b included: with a random dK it is an ordinary column sum).

Each case runs both output routes the library offers -- `grads_out` given, and `grads_out = NULL` followed by
`cast_reduce_partials_batch` over `cast_block_bwd_parts(N, which)` partials, as the engine does -- and requires them to
be bit-identical.  Row outputs sit in buffers with sentinel rows past N that must stay untouched; the ffn kernel must
give padding rows (ids == 0) exactly 0; `dx` of the qkv kernels is compared on live and on padding rows separately
(a padding row is all zero, its LayerNorm rstd is 1/sqrt(eps) = 1e4, and its gradient would otherwise set the scale).

Tolerance: 2e-5 of each tensor's max magnitude (3xTF32 products, fp32 accumulation) at every N, up to ~1e5 rows.
Largest relative errors observed over the whole GPU matrix (NVIDIA B200, 1000 W power limit): ffn dy 9.8e-7, ffn
parameter gradients 4.1e-6 (at N = 99999); qkv dx 9.3e-7 on live rows and 6.5e-7 on padding rows, qkv parameter
gradients 6.4e-6 (at N = 99999); embed dx 9.3e-7.  The gradient error grows with the rows each CTA accumulates in
fp32 (~700 at N = 99999) and stays 3x inside the bound there, so the ~1e5-row case needs no wider one.  The module
prints its maxima, with the shape where each occurred, at teardown.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from helpers import WorstErrors, backend, rel_err

EPS = 1e-8
SEED = 1234
SITE_H, SITE_O, SITE_EMB = 12, 13, 3
TOL = 2e-5
SENT = 12345.0        # fill of rows / elements past the outputs' end
EXTRA = 67            # sentinel rows after the N rows of dy / dx (longer than a tile's worth of over-write)
T = 50                # sequence length of the left-padded batches

FFN_NAMES = ("ln2.beta", "ln2.gamma", "ffn1.w", "ffn1.b", "ffn2.w", "ffn2.b")
QKV_NAMES = ("ln1.beta", "ln1.gamma", "q.w", "q.b", "k.w", "k.b", "v.w", "v.b")

WORST = WorstErrors("test_block_bwd")
_note = WORST.note


@pytest.fixture(scope="module", autouse=True)
def _report_worst(request):
    yield
    WORST.report(request.config)


def _stream(kind, dev):
    return torch.cuda.current_stream(dev).cuda_stream if kind == "gpu" else None


def padded_ids(N, rng):
    """ids of left-padded sequences of length T (the last one may be shorter): each starts with a random number of
    padding rows (id 0) and ends with at least one item."""
    ids = rng.randint(1, 1000, N).astype(np.int32)
    for s in range(0, N, T):
        n = min(T, N - s)
        ids[s:s + rng.randint(0, n)] = 0
    return ids


def ln64(x, gamma, beta):
    mu = x.mean(1, keepdim=True)
    var = ((x - mu) ** 2).mean(1, keepdim=True)
    rs = 1.0 / torch.sqrt(var + EPS)
    return gamma * ((x - mu) * rs) + beta, mu[:, 0], rs[:, 0]


class Ctx:
    def __init__(self, kind, N, H, seed):
        self.kind, self.N, self.H = kind, N, H
        self.lib, self.dev = backend(kind)
        self.st = _stream(kind, self.dev)
        self.rng = np.random.RandomState(seed)
        self.step = torch.tensor([5], dtype=torch.int64, device=self.dev)
        self.alive = []

    def randn(self, *shape, s=1.0):
        return (s * self.rng.randn(*shape)).astype(np.float32)

    def d(self, a):
        """device copy, kept alive with the context (kernels get bare pointers and run asynchronously)"""
        t = torch.from_numpy(np.ascontiguousarray(a)).to(self.dev)
        self.alive.append(t)
        return t

    def rows(self):
        """row output with EXTRA sentinel rows past N"""
        return torch.full((self.N + EXTRA, self.H), SENT, dtype=torch.float32, device=self.dev)

    def grads(self, count):
        return torch.full((count + 16,), SENT, dtype=torch.float32, device=self.dev)

    def workspace(self):
        nb = self.lib.cast_block_bwd_workspace_bytes(self.N, self.H)
        # NaN-filled: a partial the kernel fails to write poisons the reduced gradient
        return torch.full((nb // 4,), float("nan"), dtype=torch.float32, device=self.dev), nb

    def keep(self, rate, site):
        """dropout multiplier (0 or 1/(1-rate)) of every element of an [N, H] tensor, float64"""
        if rate == 0:
            return np.ones((self.N, self.H))
        k = torch.empty(self.N * self.H, dtype=torch.uint8, device=self.dev)
        assert self.lib.cast_dropout_keep(rate, SEED, self.step.data_ptr(), site, self.N * self.H, k.data_ptr(),
                                          self.st) == 0
        return k.cpu().numpy().reshape(self.N, self.H).astype(np.float64) / (1.0 - rate)

    def reduce(self, ws, which, count, out):
        parts = self.lib.cast_block_bwd_parts(self.N, which)
        assert 1 <= parts and parts * count * 4 <= ws.numel() * 4
        rc = self.lib.cast_reduce_partials_batch(1, (C.c_void_p * 1)(ws.data_ptr()), (C.c_int * 1)(parts),
                                                 (C.c_long * 1)(count), (C.c_long * 1)(count),
                                                 (C.c_void_p * 1)(out.data_ptr()), self.st)
        assert rc == 0, self.lib.cast_last_error_string()

    def two_routes(self, launch, which, count):
        """launch(rows_out, grads_out_ptr, ws, ws_bytes) both ways; returns (rows [N+EXTRA, H], grads [count]) after
        checking the routes agree bit for bit and the sentinels survived"""
        rows_a, g_a = self.rows(), self.grads(count)
        ws_a, nb = self.workspace()
        rc = launch(rows_a, g_a.data_ptr(), ws_a, nb)
        assert rc == 0, self.lib.cast_last_error_string()
        rows_b, g_b = self.rows(), self.grads(count)
        ws_b, nb = self.workspace()
        rc = launch(rows_b, None, ws_b, nb)
        assert rc == 0, self.lib.cast_last_error_string()
        self.reduce(ws_b, which, count, g_b)
        rows_a, rows_b, g_a, g_b = rows_a.cpu(), rows_b.cpu(), g_a.cpu(), g_b.cpu()
        assert torch.equal(rows_a, rows_b), "row output differs between the grads_out and the partials route"
        assert torch.equal(g_a, g_b), "gradients differ between the grads_out and the partials route"
        assert bool((rows_a[self.N:] == SENT).all()), "rows past N were written"
        assert bool((g_a[count:] == SENT).all()), "grads_out written past its end"
        return rows_a.numpy(), g_a[:count].numpy()

    def check_grads(self, kernel, got, refs, names):
        off = 0
        for name, r in zip(names, refs):
            r = r.detach().numpy().reshape(-1)
            seg = got[off:off + r.size]
            off += r.size
            e = _note(self.kind, kernel, "grads", rel_err(seg, r), f"N={self.N} H={self.H}")
            assert e <= TOL, (name, e)
        assert off == got.size


def run_ffn(kind, N, H, rate, seed=0):
    c = Ctx(kind, N, H, seed)
    lib = c.lib
    ids = padded_ids(N, c.rng)
    live = ids != 0
    W1, W2 = c.randn(H, H, s=1 / np.sqrt(H)), c.randn(H, H, s=1 / np.sqrt(H))
    b1, b2, beta = c.randn(H, s=0.1), c.randn(H, s=0.1), c.randn(H, s=0.1)
    gamma = 1 + c.randn(H, s=0.1)
    y = c.randn(N, H)             # attention output + residual: not zero on padding rows
    dx = c.randn(N, H)
    kh, ko = c.keep(rate, SITE_H), c.keep(rate, SITE_O)

    v = {k: torch.tensor(a, dtype=torch.float64, requires_grad=True)
         for k, a in (("y", y), ("gamma", gamma), ("beta", beta), ("W1", W1), ("b1", b1), ("W2", W2), ("b2", b2))}
    zn, mu, rs = ln64(v["y"], v["gamma"], v["beta"])
    h1d = torch.relu(zn @ v["W1"] + v["b1"]) * torch.from_numpy(kh)
    xout = ((h1d @ v["W2"] + v["b2"]) * torch.from_numpy(ko) + zn) * torch.from_numpy(live.astype(np.float64))[:, None]
    xout.backward(torch.from_numpy(dx.astype(np.float64)))

    f32 = lambda t: c.d(t.detach().numpy().astype(np.float32))  # noqa: E731
    dev_in = [c.d(dx), c.d(ids), f32(zn), f32(h1d), c.d(y), f32(mu), f32(rs), c.d(gamma), c.d(W1), c.d(W2)]
    ptrs = [t.data_ptr() for t in dev_in]

    def launch(out, gp, ws, nb):
        return lib.cast_ffn_bwd(*ptrs, rate, SEED, c.step.data_ptr(), SITE_O, N, H, out.data_ptr(), gp, ws.data_ptr(),
                                nb, c.st)

    count = 2 * H + 2 * (H * H + H)
    rows, g = c.two_routes(launch, 0, count)
    dy = rows[:N]
    assert (dy[~live] == 0).all(), "padding rows must get exactly 0 from cast_ffn_bwd"
    e = _note(kind, "ffn", "dy", rel_err(dy, v["y"].grad.numpy()), f"N={N} H={H}")
    assert e <= TOL, e
    c.check_grads("ffn", g, [v[k].grad for k in ("beta", "gamma", "W1", "b1", "W2", "b2")], FFN_NAMES)


def run_qkv(kind, N, H, rate, seed=0):
    """cast_qkv_bwd, then cast_qkv_bwd_embed with dropout rate `rate` on the same inputs"""
    c = Ctx(kind, N, H, seed)
    lib = c.lib
    ids = padded_ids(N, c.rng)
    live = ids != 0
    W = {k: c.randn(H, H, s=1 / np.sqrt(H)) for k in ("q", "k", "v")}
    b = {k: c.randn(H, s=0.1) for k in ("q", "k", "v")}
    gamma, beta = 1 + c.randn(H, s=0.1), c.randn(H, s=0.1)
    x = c.randn(N, H)
    x[~live] = 0.0                # block input of a padding position is exactly zero (the previous block's mask)
    dQ, dK, dV, dres = (c.randn(N, H) for _ in range(4))

    v = {k: torch.tensor(a, dtype=torch.float64, requires_grad=True)
         for k, a in (("x", x), ("gamma", gamma), ("beta", beta), ("Wq", W["q"]), ("bq", b["q"]), ("Wk", W["k"]),
                      ("bk", b["k"]), ("Wv", W["v"]), ("bv", b["v"]))}
    qn, mu, rs = ln64(v["x"], v["gamma"], v["beta"])
    t64 = lambda a: torch.from_numpy(a.astype(np.float64))  # noqa: E731
    loss = ((qn @ v["Wq"] + v["bq"]) * t64(dQ)).sum() + ((v["x"] @ v["Wk"] + v["bk"]) * t64(dK)).sum() \
        + ((v["x"] @ v["Wv"] + v["bv"]) * t64(dV)).sum() + (qn * t64(dres)).sum()
    loss.backward()
    ref_dx = v["x"].grad.numpy()
    ref_g = [v[k].grad for k in ("beta", "gamma", "Wq", "bq", "Wk", "bk", "Wv", "bv")]

    f32 = lambda t: c.d(t.detach().numpy().astype(np.float32))  # noqa: E731
    dev_in = [c.d(dQ), c.d(dK), c.d(dV), c.d(dres), c.d(x), f32(qn), f32(mu), f32(rs), c.d(gamma), c.d(W["q"]),
              c.d(W["k"]), c.d(W["v"])]
    ptrs = [t.data_ptr() for t in dev_in]
    count = 2 * H + 3 * (H * H + H)

    def check_dx(kernel, got, ref):
        for part, sel in (("dx live", live), ("dx padding", ~live)):
            if sel.any():
                e = _note(kind, kernel, part, rel_err(got[sel], ref[sel]), f"N={N} H={H}")
                assert e <= TOL, (part, e)

    def launch(out, gp, ws, nb):
        return lib.cast_qkv_bwd(*ptrs, N, H, out.data_ptr(), gp, ws.data_ptr(), nb, c.st)

    rows, g = c.two_routes(launch, 1, count)
    check_dx("qkv", rows[:N], ref_dx)
    c.check_grads("qkv", g, ref_g, QKV_NAMES)

    d_ids = c.d(ids)

    def launch_embed(out, gp, ws, nb):
        return lib.cast_qkv_bwd_embed(*ptrs, N, H, d_ids.data_ptr(), rate, SEED, c.step.data_ptr(), SITE_EMB,
                                      out.data_ptr(), gp, ws.data_ptr(), nb, c.st)

    rows_e, g_e = c.two_routes(launch_embed, 1, count)
    assert np.array_equal(g_e, g), "the embed variant's parameter gradients must be cast_qkv_bwd's"
    ref_e = ref_dx * live[:, None] * c.keep(rate, SITE_EMB)
    dx_e = rows_e[:N]
    assert (dx_e[~live] == 0).all()
    e = _note(kind, "embed", "dx", rel_err(dx_e[live], ref_e[live]), f"N={N} H={H}")
    assert e <= TOL, e
    if rate > 0:
        assert ((dx_e == 0) == (ref_e == 0)).all(), "dropped elements differ"


def run_arg_checks(kind):
    """documented error codes, returned before anything is launched; outputs untouched"""
    N, H = 100, 16
    lib, dev = backend(kind)
    st = _stream(kind, dev)
    buf = lambda n: torch.zeros(n, dtype=torch.float32, device=dev)  # noqa: E731
    a = buf(N * 65)                           # big enough for every operand below
    w = buf(65 * 65)
    ids = torch.ones(N, dtype=torch.int32, device=dev)
    out = torch.full((N * 65,), SENT, dtype=torch.float32, device=dev)
    g = torch.full((3 * 65 * 66 + 130,), SENT, dtype=torch.float32, device=dev)
    ws = buf(lib.cast_block_bwd_workspace_bytes(25600, 65) // 4)
    step = torch.zeros(1, dtype=torch.int64, device=dev)
    p = a.data_ptr()

    def ffn(n, h, nb):
        return lib.cast_ffn_bwd(p, ids.data_ptr(), p, p, p, p, p, p, w.data_ptr(), w.data_ptr(), 0.1, SEED,
                                step.data_ptr(), SITE_O, n, h, out.data_ptr(), g.data_ptr(), ws.data_ptr(), nb, st)

    def qkv(n, h, nb):
        return lib.cast_qkv_bwd(p, p, p, p, p, p, p, p, p, w.data_ptr(), w.data_ptr(), w.data_ptr(), n, h,
                                out.data_ptr(), g.data_ptr(), ws.data_ptr(), nb, st)

    def emb(n, h, nb):
        return lib.cast_qkv_bwd_embed(p, p, p, p, p, p, p, p, p, w.data_ptr(), w.data_ptr(), w.data_ptr(), n, h,
                                      ids.data_ptr(), 0.1, SEED, step.data_ptr(), SITE_EMB, out.data_ptr(),
                                      g.data_ptr(), ws.data_ptr(), nb, st)

    full = ws.numel() * 4
    for call in (ffn, qkv, emb):
        n0 = lib.cast_launch_count()
        need = lib.cast_block_bwd_workspace_bytes(N, H)
        assert call(N, H, need - 4) == -3                  # CAST_ERR_WORKSPACE
        assert call(N, 65, full) == -2                     # CAST_ERR_UNSUPPORTED
        assert call(N, 0, full) == -2
        assert call(0, H, full) == -1                      # CAST_ERR_BAD_ARG
        assert call(-1, H, full) == -1
        assert lib.cast_launch_count() == n0, "a rejected call launched a kernel"
    assert bool((out.cpu() == SENT).all()) and bool((g.cpu() == SENT).all())
    # and a null workspace is a workspace error, not a fault
    assert lib.cast_ffn_bwd(p, ids.data_ptr(), p, p, p, p, p, p, w.data_ptr(), w.data_ptr(), 0.1, SEED,
                            step.data_ptr(), SITE_O, N, H, out.data_ptr(), g.data_ptr(), None, full, st) == -3
    assert lib.cast_qkv_bwd(p, p, p, p, p, p, p, p, p, w.data_ptr(), w.data_ptr(), w.data_ptr(), N, H,
                            out.data_ptr(), g.data_ptr(), None, full, st) == -3


# ---------------------------------------------------------------------------------------------------- emulated
EMU_CASES = [(1, 7, 0.2), (63, 13, 0.0), (64, 8, 0.3), (65, 16, 0.2), (130, 33, 0.25), (129, 24, 0.0),
             (70, 50, 0.2), (100, 63, 0.2), (150, 64, 0.1)]


@pytest.mark.emu
@pytest.mark.parametrize("N,H,rate", EMU_CASES)
def test_ffn_bwd_emulated(N, H, rate):
    run_ffn("emu", N, H, rate)


@pytest.mark.emu
@pytest.mark.parametrize("N,H,rate", EMU_CASES)
def test_qkv_bwd_emulated(N, H, rate):
    run_qkv("emu", N, H, rate)


@pytest.mark.emu
def test_block_bwd_emulated_second_tile():
    """9473 rows = 148 one-tile CTAs plus a one-row 149th tile that CTA 0 walks second (fixed 148-CTA grid)"""
    run_ffn("emu", 9473, 7, 0.2)
    run_qkv("emu", 9473, 7, 0.2)


@pytest.mark.emu
def test_block_bwd_arg_checks_emulated():
    run_arg_checks("emu")


# ---------------------------------------------------------------------------------------------------------- GPU
# one H per KS instance (8 .. 64) plus H that are not multiples of 8 or 2 (scalar cp.async, unpaired dx stores);
# N: partial tiles, 9472 = 148 * 64 (one tile per CTA), 9473 (a second one-row tile), 2 * 9472 + 1, BASELINE C2, ~1e5
GPU_H = [7, 8, 13, 16, 24, 32, 33, 40, 48, 49, 50, 56, 63, 64]
GPU_N = [1, 63, 64, 65, 800, 9472, 9473, 2 * 9472 + 1, 25600, 99999]


@pytest.mark.gpu
@pytest.mark.parametrize("rate", [0.0, 0.2])
@pytest.mark.parametrize("N", GPU_N)
@pytest.mark.parametrize("H", GPU_H)
def test_ffn_bwd_gpu(H, N, rate):
    run_ffn("gpu", N, H, rate, seed=N + H)


@pytest.mark.gpu
@pytest.mark.parametrize("rate", [0.0, 0.3])
@pytest.mark.parametrize("N", GPU_N)
@pytest.mark.parametrize("H", GPU_H)
def test_qkv_bwd_gpu(H, N, rate):
    run_qkv("gpu", N, H, rate, seed=N + H)


@pytest.mark.gpu
def test_block_bwd_arg_checks_gpu():
    run_arg_checks("gpu")
