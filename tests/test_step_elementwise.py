"""The small kernels of every training step, each against a plain restatement of its formula (include/cast_b200.h):

* `cast_layernorm_fwd` -- y, mean, rstd against float64 (modules.py:53-80), the zero-sum flags xnz / ynz exactly, on
  all-zero rows and rows whose sum is exactly 0 in any summation order; one H or more per template instance
  (NV = 2, 4, 8, 16, 32 values per lane);
* `cast_layernorm_bwd` -- dx (with and without dx_add), dgamma and dbeta against float64 autograd; dgamma / dbeta
  through the reduced route and through the partials left in the workspace (`cast_reduce_partials_batch` with pitch
  2H), which must agree bit for bit;
* `cast_embed_fwd` -- the gather, position row n % T, context add, dropout and padding mask against numpy fp32 in
  the kernel's order of operations, bit for bit (a power-of-two scale keeps the product exact, so FMA contraction
  cannot change a bit); odd H (element index row * H + c odd, the unpaired dropout hash path), ids 0 and >= V,
  an unaligned output (scalar stores);
* `cast_mask_dropout`, `cast_concat_dropout_fwd` / `_bwd`, `cast_relu_bwd` -- bit for bit against numpy fp32 with
  keep masks from `cast_dropout_keep` (masking and dropout round once per element at most);
* `cast_colsum` -- against float64, with a row stride larger than the column count, odd column counts and up to
  ~1e5 rows; bit-identical across calls.

Tolerance for the reductions (LayerNorm, colsum): 2e-5 of each tensor's max magnitude (fp32 accumulation).  The
LayerNorm statistics are checked per row instead, because an all-zero row's rstd (1e4) would otherwise set the scale:
rstd within 2e-5 of each row's value, mean within 2e-6 of each row's mean |x|.  Largest relative errors observed
(NVIDIA B200, 1000 W power limit): layernorm_fwd y 1.9e-7, rstd 1.8e-7 and mean 1.7e-7 per row; layernorm_bwd dx
2.0e-7, dgamma 4.3e-7, dbeta 1.6e-7; colsum 5.3e-7.  The module prints its maxima, with the shape where each occurred,
at teardown.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from helpers import WorstErrors, backend, rel_err

SEED = 777
TOL = 2e-5
SENT = 12345.0

WORST = WorstErrors("test_step_elementwise")
_note = WORST.note


@pytest.fixture(scope="module", autouse=True)
def _report_worst(request):
    yield
    WORST.report(request.config)


class Ctx:
    def __init__(self, kind, seed):
        self.kind = kind
        self.lib, self.dev = backend(kind)
        self.st = torch.cuda.current_stream(self.dev).cuda_stream if kind == "gpu" else None
        self.rng = np.random.RandomState(seed)
        self.step = torch.tensor([9], dtype=torch.int64, device=self.dev)
        self.alive = []

    def d(self, a):
        """device copy, kept alive with the context: the callers pass bare pointers to kernels that run asynchronously,
        and a temporary freed after `.data_ptr()` would hand its memory to the next operand"""
        t = torch.from_numpy(np.ascontiguousarray(a)).to(self.dev)
        self.alive.append(t)
        return t

    def full(self, *shape, v=SENT):
        return torch.full(shape, v, dtype=torch.float32, device=self.dev)

    def mult(self, rate, site, n):
        """fp32 dropout multipliers of elements 0..n-1 of a site: 0 or float32(1 / (1 - rate)), as kernels form them"""
        if rate == 0 or n == 0:
            return np.ones(n, np.float32)
        k = torch.empty(n, dtype=torch.uint8, device=self.dev)
        assert self.lib.cast_dropout_keep(rate, SEED, self.step.data_ptr(), site, n, k.data_ptr(), self.st) == 0
        scale = np.float32(1.0) / (np.float32(1.0) - np.float32(rate))
        return np.where(k.cpu().numpy() != 0, scale, np.float32(0.0)).astype(np.float32)


def exact_zero_sum(rng, H, scale=16.0):
    """H dyadic values (multiples of 1/scale) in +/- pairs: every partial sum is exact, so the sum is 0 in any order"""
    v = rng.randint(-64, 65, H // 2).astype(np.float32) / np.float32(scale)
    row = np.concatenate([v, -v, np.zeros(H % 2, np.float32)])
    return rng.permutation(row).astype(np.float32)


# ------------------------------------------------------------------------------------------------ LayerNorm
def ln_inputs(c, N, H, zero_sum_beta):
    x = (c.rng.randn(N, H) + 0.5 * c.rng.randn(N, 1)).astype(np.float32)
    kinds = np.zeros(N, np.int32)                       # 0 random, 1 all zero, 2 sum exactly zero
    for r in range(1, N, 5):
        x[r] = 0.0
        kinds[r] = 1
    for r in range(3, N, 5):
        x[r] = exact_zero_sum(c.rng, H)
        kinds[r] = 2
    gamma = (1 + 0.1 * c.rng.randn(H)).astype(np.float32)
    beta = exact_zero_sum(c.rng, H, 64.0) if zero_sum_beta else (0.3 + 0.1 * c.rng.randn(H)).astype(np.float32)
    return x, gamma, beta, kinds


def run_layernorm_fwd(kind, N, H, zero_sum_beta):
    c = Ctx(kind, N * 1000 + H)
    x, gamma, beta, kinds = ln_inputs(c, N, H, zero_sum_beta)
    y, mean, rstd, xnz, ynz = c.full(N + 3, H), c.full(N + 3), c.full(N + 3), c.full(N + 3), c.full(N + 3)
    rc = c.lib.cast_layernorm_fwd(c.d(x).data_ptr(), c.d(gamma).data_ptr(), c.d(beta).data_ptr(), N, H, 1e-8,
                                  y.data_ptr(), mean.data_ptr(), rstd.data_ptr(), xnz.data_ptr(), ynz.data_ptr(), c.st)
    assert rc == 0, c.lib.cast_last_error_string()
    y, mean, rstd, xnz, ynz = (t.cpu().numpy() for t in (y, mean, rstd, xnz, ynz))
    for t in (y, mean, rstd, xnz, ynz):
        assert (t[N:] == SENT).all(), "written past row N"
    x64 = x.astype(np.float64)
    mu = x64.mean(1)
    rs = 1.0 / np.sqrt(((x64 - mu[:, None]) ** 2).mean(1) + 1e-8)
    yr = gamma * ((x64 - mu[:, None]) * rs[:, None]) + beta
    assert _note(kind, "layernorm_fwd", "y", rel_err(y[:N], yr), f"N={N} H={H}") <= TOL
    # The statistics are checked row by row, not against the tensor's max: an all-zero row has rstd = 1/sqrt(eps)
    # = 1e4, which would make a max-relative bound 0.2 absolute on ordinary rows (rstd ~ 1).  rstd > 0, so its error
    # is relative per row; the error of mean is taken relative to the row's mean |x| (what an fp32 sum's error scales
    # with), and mean is exactly 0 on the all-zero and zero-sum rows.
    rs_err = float((np.abs(rstd[:N].astype(np.float64) - rs) / rs).max())
    assert _note(kind, "layernorm_fwd", "rstd (per row)", rs_err, f"N={N} H={H}") <= TOL
    live = kinds == 0
    if live.any():
        mu_err = float((np.abs(mean[:N][live] - mu[live]) / np.abs(x64[live]).mean(1)).max())
        assert _note(kind, "layernorm_fwd", "mean (per row)", mu_err, f"N={N} H={H}") <= 2e-6
    assert (mean[:N][kinds > 0] == 0).all()
    assert np.array_equal(xnz[:N], (kinds == 0).astype(np.float32))    # random rows never sum to exactly 0
    # all-zero rows: y = beta exactly, so ynz = (sum(beta) != 0); elsewhere compare where the sum is clearly not 0
    assert (y[:N][kinds == 1] == beta).all()
    ys = yr.sum(1)
    zero_rows = kinds == 1
    assert (ynz[:N][zero_rows] == (0.0 if zero_sum_beta else 1.0)).all()
    clear = ~zero_rows & (np.abs(ys) > 1e-3)
    assert np.array_equal(ynz[:N][clear], np.ones(int(clear.sum()), np.float32))


def run_layernorm_bwd(kind, N, H, with_add):
    c = Ctx(kind, N * 1000 + H + 1)
    lib = c.lib
    x = (c.rng.randn(N, H) + 0.5 * c.rng.randn(N, 1)).astype(np.float32)
    gamma = (1 + 0.1 * c.rng.randn(H)).astype(np.float32)
    dy = c.rng.randn(N, H).astype(np.float32)
    add = c.rng.randn(N, H).astype(np.float32) if with_add else None
    xv = torch.tensor(x, dtype=torch.float64, requires_grad=True)
    gv = torch.tensor(gamma, dtype=torch.float64, requires_grad=True)
    bv = torch.zeros(H, dtype=torch.float64, requires_grad=True)
    mu = xv.mean(1, keepdim=True)
    rs = 1.0 / torch.sqrt(((xv - mu) ** 2).mean(1, keepdim=True) + 1e-8)
    (gv * ((xv - mu) * rs) + bv).backward(torch.from_numpy(dy.astype(np.float64)))
    ref_dx = xv.grad.numpy() + (add if with_add else 0.0)
    f32 = lambda t: c.d(t.detach().numpy().reshape(-1).astype(np.float32))  # noqa: E731
    ins = [c.d(dy), c.d(x), f32(mu), f32(rs), c.d(gamma)]
    d_add = c.d(add) if with_add else None
    nb = lib.cast_layernorm_bwd_workspace_bytes(N, H)
    parts = lib.cast_layernorm_bwd_parts(N)
    assert nb == parts * 2 * H * 4

    def launch(dg, db):
        dx = c.full(N + 2, H)
        ws = c.full(nb // 4, v=float("nan"))
        rc = lib.cast_layernorm_bwd(*[t.data_ptr() for t in ins], N, H, d_add.data_ptr() if with_add else None,
                                    dx.data_ptr(), dg, db, ws.data_ptr(), nb, c.st)
        assert rc == 0, lib.cast_last_error_string()
        return dx, ws

    dgam, dbet = c.full(H + 1), c.full(H + 1)
    dx_a, _ = launch(dgam.data_ptr(), dbet.data_ptr())
    dx_b, ws = launch(None, None)
    dgam_b, dbet_b = c.full(H + 1), c.full(H + 1)
    base = ws.data_ptr()
    rc = lib.cast_reduce_partials_batch(2, (C.c_void_p * 2)(base, base + 4 * H), (C.c_int * 2)(parts, parts),
                                        (C.c_long * 2)(H, H), (C.c_long * 2)(2 * H, 2 * H),
                                        (C.c_void_p * 2)(dgam_b.data_ptr(), dbet_b.data_ptr()), c.st)
    assert rc == 0, lib.cast_last_error_string()
    dx_a, dx_b, dgam, dbet, dgam_b, dbet_b = (t.cpu() for t in (dx_a, dx_b, dgam, dbet, dgam_b, dbet_b))
    assert torch.equal(dx_a, dx_b) and torch.equal(dgam, dgam_b) and torch.equal(dbet, dbet_b)
    assert bool((dx_a[N:] == SENT).all()) and float(dgam[H]) == SENT and float(dbet[H]) == SENT
    assert _note(kind, "layernorm_bwd", "dx", rel_err(dx_a[:N].numpy(), ref_dx), f"N={N} H={H}") <= TOL
    assert _note(kind, "layernorm_bwd", "dgamma", rel_err(dgam[:H].numpy(), gv.grad.numpy()), f"N={N} H={H}") <= TOL
    assert _note(kind, "layernorm_bwd", "dbeta", rel_err(dbet[:H].numpy(), bv.grad.numpy()), f"N={N} H={H}") <= TOL


# ------------------------------------------------------------------------------------------------ embedding
def run_embed_fwd(kind, N, H, T, V, rate, use_pos, use_add, use_mask, scale=2.0, misalign=False):
    c = Ctx(kind, N * 7 + H)
    site = 5
    table = c.rng.randn(V, H).astype(np.float32)
    table[0] = 0.0
    ids = c.rng.randint(1, V, N).astype(np.int32)
    ids[:: 4] = 0                                    # padding
    ids[1:: 9] = V                                   # out of range: treated as padding
    ids[2:: 11] = V + 17
    pos = c.rng.randn(T, H).astype(np.float32)
    add = c.rng.randn(N, H).astype(np.float32)
    mask_ids = (c.rng.rand(N) > 0.3).astype(np.int32) * c.rng.randint(1, 50, N).astype(np.int32)
    off = 1 if misalign else 0
    out = c.full(N * H + off + H)
    rc = c.lib.cast_embed_fwd(c.d(ids).data_ptr(), c.d(table).data_ptr(), V, H, N, T, scale,
                              c.d(pos).data_ptr() if use_pos else None, c.d(add).data_ptr() if use_add else None,
                              rate, SEED, c.step.data_ptr(), site, c.d(mask_ids).data_ptr() if use_mask else None,
                              out.data_ptr() + 4 * off, c.st)
    assert rc == 0, c.lib.cast_last_error_string()
    got = out.cpu().numpy()
    assert (got[:off] == SENT).all() and (got[off + N * H:] == SENT).all()
    got = got[off:off + N * H].reshape(N, H)
    live = (ids > 0) & (ids < V)
    s = np.float32(scale)
    v = np.where(live[:, None], table[np.where(live, ids, 0)] * s, np.float32(0.0)).astype(np.float32)
    if use_pos:
        v = (v + pos[np.arange(N) % T]).astype(np.float32)
    if use_add:
        v = (v + add).astype(np.float32)
    v = (v * c.mult(rate, site, N * H).reshape(N, H)).astype(np.float32)
    m = (mask_ids != 0).astype(np.float32) if use_mask else np.ones(N, np.float32)
    v = (v * m[:, None]).astype(np.float32)
    if np.log2(scale) == int(np.log2(scale)):
        assert np.array_equal(got, v)
    else:  # an inexact product may be fused with the add that follows it: one rounding less
        assert (got == 0).sum() == (v == 0).sum() and np.array_equal(got == 0, v == 0)
        assert _note(kind, "embed_fwd", "out (sqrt(H) scale)", rel_err(got, v)) <= 1e-6


# --------------------------------------------------------------------------------------- masks and dropout
def run_mask_dropout(kind, N, H, rate):
    c = Ctx(kind, N + H)
    site = 21
    x = c.rng.randn(N, H).astype(np.float32)
    ids = (c.rng.rand(N) > 0.3).astype(np.int32) * c.rng.randint(1, 50, N).astype(np.int32)
    m = (ids != 0).astype(np.float32)[:, None]
    ref_m = (x * m).astype(np.float32)
    ref_md = (ref_m * c.mult(rate, site, N * H).reshape(N, H)).astype(np.float32)
    dx, di = c.d(x), c.d(ids)
    for want_m, want_md in ((True, True), (True, False), (False, True)):
        om, omd = c.full(N + 1, H), c.full(N + 1, H)
        rc = c.lib.cast_mask_dropout(dx.data_ptr(), di.data_ptr(), rate, SEED, c.step.data_ptr(), site, N, H,
                                     om.data_ptr() if want_m else None, omd.data_ptr() if want_md else None, c.st)
        assert rc == 0, c.lib.cast_last_error_string()
        om, omd = om.cpu().numpy(), omd.cpu().numpy()
        assert np.array_equal(om[:N], ref_m) if want_m else (om == SENT).all()
        assert np.array_equal(omd[:N], ref_md) if want_md else (omd == SENT).all()
        assert (om[N:] == SENT).all() and (omd[N:] == SENT).all()
    # no mask: dropout only
    omd = c.full(N, H)
    rc = c.lib.cast_mask_dropout(dx.data_ptr(), None, rate, SEED, c.step.data_ptr(), site, N, H, None, omd.data_ptr(),
                                 c.st)
    assert rc == 0
    assert np.array_equal(omd.cpu().numpy(), (x * c.mult(rate, site, N * H).reshape(N, H)).astype(np.float32))


def run_concat(kind, N, H, k, wa, rate_a, rate_b):
    c = Ctx(kind, N * 31 + H * 5 + k * 3 + wa)
    site_a, site_b = 41, 42
    srcs = [c.rng.randn(N, H).astype(np.float32) for _ in range(k)]
    mA = c.mult(rate_a, site_a, N * wa * H).reshape(N, wa * H)
    mB = c.mult(rate_b, site_b, N * k * H).reshape(N, k * H)
    cat = np.concatenate(srcs, 1)
    ref = cat.copy()
    ref[:, :wa * H] = (ref[:, :wa * H] * mA).astype(np.float32)
    ref = (ref * mB).astype(np.float32)
    d_srcs = [c.d(s) for s in srcs]
    out = c.full(N * k * H + 5)
    rc = c.lib.cast_concat_dropout_fwd((C.c_void_p * k)(*[s.data_ptr() for s in d_srcs]), k, wa, N, H, rate_a, site_a,
                                       rate_b, site_b, SEED, c.step.data_ptr(), out.data_ptr(), c.st)
    assert rc == 0, c.lib.cast_last_error_string()
    got = out.cpu().numpy()
    assert np.array_equal(got[:N * k * H].reshape(N, k * H), ref) and (got[N * k * H:] == SENT).all()
    # backward: the same multipliers on the gradient, split back into the sources; the last destination is null
    dcat = c.rng.randn(N, k * H).astype(np.float32)
    gref = dcat.copy()
    gref[:, :wa * H] = (gref[:, :wa * H] * mA).astype(np.float32)
    gref = (gref * mB).astype(np.float32)
    dsts = [c.full(N + 1, H) for _ in range(k)]
    ptrs = [d.data_ptr() for d in dsts]
    if k > 1:
        ptrs[-1] = None
    rc = c.lib.cast_concat_dropout_bwd(c.d(dcat).data_ptr(), k, wa, N, H, rate_a, site_a, rate_b, site_b, SEED,
                                       c.step.data_ptr(), (C.c_void_p * k)(*ptrs), c.st)
    assert rc == 0, c.lib.cast_last_error_string()
    for s in range(k):
        g = dsts[s].cpu().numpy()
        if ptrs[s] is None:
            assert (g == SENT).all()
        else:
            assert np.array_equal(g[:N], gref[:, s * H:(s + 1) * H]) and (g[N:] == SENT).all(), s


def run_relu_bwd(kind, n, scale):
    c = Ctx(kind, n)
    dy = c.rng.randn(n).astype(np.float32)
    act = c.rng.randn(n).astype(np.float32)
    act[::5] = 0.0
    act[1::7] = -0.0
    # subnormal activations: active when positive under IEEE comparison; the library is built without flush-to-zero
    # (build.py passes neither --use_fast_math nor -ftz=true), and a flush-to-zero build would treat them as 0
    act[2::11] = np.float32(1e-40)
    act[3::13] = np.float32(-1e-40)
    out = c.full(n + 3)
    assert c.lib.cast_relu_bwd(c.d(dy).data_ptr(), c.d(act).data_ptr(), scale, out.data_ptr(), n, c.st) == 0
    got = out.cpu().numpy()
    ref = np.where(act > 0, (dy * np.float32(scale)).astype(np.float32), np.float32(0.0))
    # array_equal treats +0 and -0 as equal: the header's dy * 0 for an inactive unit may carry dy's sign
    assert np.array_equal(got[:n], ref) and (got[n:] == SENT).all()


# ------------------------------------------------------------------------------------------------ colsum
def run_colsum(kind, rows, cols, ld):
    c = Ctx(kind, rows + cols + ld)
    X = (c.rng.randn(rows, ld) + 0.3).astype(np.float32)
    X[:, cols:] = np.float32(1e30)                   # stride padding must not be read into the sums
    nb = c.lib.cast_colsum_workspace_bytes(rows, cols)
    dX = c.d(X)
    outs = []
    for _ in range(2):
        out = c.full(cols + 2)
        ws = c.full(nb // 4, v=float("nan"))
        rc = c.lib.cast_colsum(dX.data_ptr(), rows, cols, ld, out.data_ptr(), ws.data_ptr(), nb, c.st)
        assert rc == 0, c.lib.cast_last_error_string()
        outs.append(out.cpu().numpy())
    assert np.array_equal(outs[0], outs[1])
    assert (outs[0][cols:] == SENT).all()
    ref = X[:, :cols].astype(np.float64).sum(0)
    assert _note(kind, "colsum", "out", rel_err(outs[0][:cols], ref), f"rows={rows} cols={cols}") <= TOL


# ---------------------------------------------------------------------------------------------------- emulated
@pytest.mark.emu
@pytest.mark.parametrize("N,H", [(19, 7), (13, 64), (11, 65), (9, 129), (7, 257), (5, 1000)])
def test_layernorm_fwd_emulated(N, H):
    run_layernorm_fwd("emu", N, H, zero_sum_beta=H % 2 == 1)


@pytest.mark.emu
@pytest.mark.parametrize("N,H,with_add", [(70, 7, True), (130, 50, False), (65, 128, True), (33, 129, False),
                                          (20, 300, True), (9, 1024, False)])
def test_layernorm_bwd_emulated(N, H, with_add):
    run_layernorm_bwd("emu", N, H, with_add)


EMBED_CASES = [  # N, H, T, V, rate, pos, add, mask
    (40, 7, 10, 30, 0.3, True, True, True), (40, 50, 10, 30, 0.3, True, True, True),
    (33, 13, 50, 20, 0.0, True, False, True), (33, 64, 7, 20, 0.25, False, True, False),
    (25, 33, 4, 12, 0.5, True, True, False), (30, 1, 5, 9, 0.2, True, False, True)]


@pytest.mark.emu
@pytest.mark.parametrize("N,H,T,V,rate,pos,add,mask", EMBED_CASES)
def test_embed_fwd_emulated(N, H, T, V, rate, pos, add, mask):
    run_embed_fwd("emu", N, H, T, V, rate, pos, add, mask)


@pytest.mark.emu
def test_embed_fwd_emulated_unaligned_and_inexact_scale():
    run_embed_fwd("emu", 40, 50, 10, 30, 0.2, True, True, True, misalign=True)
    run_embed_fwd("emu", 40, 50, 10, 30, 0.2, True, True, True, scale=float(np.sqrt(50)))


@pytest.mark.emu
@pytest.mark.parametrize("N,H,rate", [(37, 7, 0.3), (20, 50, 0.0), (64, 16, 0.5)])
def test_mask_dropout_emulated(N, H, rate):
    run_mask_dropout("emu", N, H, rate)


CONCAT_CASES = [(k, wa) for k in range(1, 5) for wa in range(0, k + 1)]


@pytest.mark.emu
@pytest.mark.parametrize("k,wa", CONCAT_CASES)
def test_concat_dropout_emulated(k, wa):
    run_concat("emu", 23, 7, k, wa, 0.3, 0.15)


@pytest.mark.emu
def test_concat_dropout_single_site_emulated():
    """the form the engine uses for its merges: width_a = 0, one dropout over the whole concatenation"""
    run_concat("emu", 30, 50, 2, 0, 0.0, 0.2)
    run_concat("emu", 30, 50, 3, 0, 0.0, 0.2)


@pytest.mark.emu
def test_relu_bwd_emulated():
    run_relu_bwd("emu", 3001, 1.0)
    run_relu_bwd("emu", 777, 1.25)


@pytest.mark.emu
@pytest.mark.parametrize("rows,cols,ld", [(1, 1, 1), (300, 33, 40), (5000, 17, 17), (4097, 129, 131)])
def test_colsum_emulated(rows, cols, ld):
    run_colsum("emu", rows, cols, ld)


# ---------------------------------------------------------------------------------------------------------- GPU
LN_H = [7, 50, 64, 65, 128, 129, 256, 257, 512, 1000, 1024]


@pytest.mark.gpu
@pytest.mark.parametrize("N", [1, 999, 25600])
@pytest.mark.parametrize("H", LN_H)
def test_layernorm_fwd_gpu(H, N):
    run_layernorm_fwd("gpu", N, H, zero_sum_beta=False)
    run_layernorm_fwd("gpu", N, H, zero_sum_beta=True)


@pytest.mark.gpu
@pytest.mark.parametrize("with_add", [False, True])
@pytest.mark.parametrize("N", [1, 999, 25600])
@pytest.mark.parametrize("H", LN_H)
def test_layernorm_bwd_gpu(H, N, with_add):
    run_layernorm_bwd("gpu", N, H, with_add)


@pytest.mark.gpu
@pytest.mark.parametrize("N,H,T,V,rate,pos,add,mask", EMBED_CASES + [
    (25600, 50, 50, 3417, 0.2, True, True, True), (25600, 49, 50, 3417, 0.2, True, True, True),
    (9999, 64, 200, 50000, 0.5, True, False, True), (1, 33, 1, 2, 0.3, True, True, True)])
def test_embed_fwd_gpu(N, H, T, V, rate, pos, add, mask):
    run_embed_fwd("gpu", N, H, T, V, rate, pos, add, mask)


@pytest.mark.gpu
def test_embed_fwd_gpu_unaligned_and_inexact_scale():
    run_embed_fwd("gpu", 2000, 50, 50, 300, 0.2, True, True, True, misalign=True)
    run_embed_fwd("gpu", 2000, 50, 50, 300, 0.2, True, True, True, scale=float(np.sqrt(50)))
    run_embed_fwd("gpu", 2000, 33, 50, 300, 0.2, True, True, True, scale=float(np.sqrt(33)))


@pytest.mark.gpu
@pytest.mark.parametrize("N,H,rate", [(25600, 50, 0.2), (999, 7, 0.3), (64, 64, 0.0), (10001, 33, 0.5)])
def test_mask_dropout_gpu(N, H, rate):
    run_mask_dropout("gpu", N, H, rate)


@pytest.mark.gpu
@pytest.mark.parametrize("k,wa", CONCAT_CASES)
@pytest.mark.parametrize("N,H", [(25600, 50), (999, 7)])
def test_concat_dropout_gpu(N, H, k, wa):
    run_concat("gpu", N, H, k, wa, 0.3, 0.15)


@pytest.mark.gpu
def test_concat_dropout_single_site_gpu():
    run_concat("gpu", 25600, 50, 2, 0, 0.0, 0.2)
    run_concat("gpu", 25600, 50, 4, 0, 0.0, 0.2)


@pytest.mark.gpu
def test_relu_bwd_gpu():
    run_relu_bwd("gpu", 25600 * 50, 1.0)
    run_relu_bwd("gpu", 12345, 1.25)


@pytest.mark.gpu
@pytest.mark.parametrize("rows,cols,ld", [(1, 1, 1), (4095, 50, 50), (4096, 33, 40), (25600, 50, 150),
                                          (99999, 129, 131), (100000, 64, 64), (777, 1000, 1003)])
def test_colsum_gpu(rows, cols, ld):
    run_colsum("gpu", rows, cols, ld)
