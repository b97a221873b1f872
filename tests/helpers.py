"""Shared test helpers: backend selection (real CUDA library on a GPU box; host-emulated kernels for CPU logic
tests), oracle hand-off of dropout masks, comparison utilities."""
import ctypes
import os
import subprocess
import sys
from types import SimpleNamespace

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import cast_b200  # noqa: E402
from cast_b200 import _lib as castlib  # noqa: E402
from oracle import cast_oracle as O  # noqa: E402

EMU_SO = os.path.join(ROOT, "tests", "emu", "_build", "libcast_emu.so")
_emu = None


def emu_lib():
    """TEST INFRASTRUCTURE: the kernel sources compiled for the host (tests/emu).  Never used by the package."""
    global _emu
    if _emu is None:
        import fcntl
        os.makedirs(os.path.dirname(EMU_SO), exist_ok=True)
        with open(EMU_SO + ".lock", "w") as lk:  # several test processes (gloo ranks) may arrive together
            fcntl.flock(lk, fcntl.LOCK_EX)
            subprocess.check_call(["bash", os.path.join(ROOT, "tests", "emu", "build_emu.sh")],
                                  stdout=subprocess.DEVNULL)
            _emu = castlib.bind(ctypes.CDLL(EMU_SO))
    return _emu


def backend(kind):
    """kind = 'gpu' -> (cuda lib, cuda device); kind = 'emu' -> (emulated lib, cpu)."""
    if kind == "gpu":
        lib = castlib.load_library()
        lib.cast_set_pdl(0)   # ABI-level tests feed kernels operands made by the launch just before: plain stream order
        return lib, torch.device("cuda", 0)
    return emu_lib(), torch.device("cpu")


def make_args(**kw):
    d = dict(hidden_units=50, maxlen=50, num_heads=1, num_blocks=2, num_context_blocks=2, max_bins=200, l2_emb=0.0,
             lr=1e-3, dropout_rate=0.0, seed=42, bin_in_hours=48, log_scale=False)
    d.update(kw)
    return SimpleNamespace(**d)


def golden_batch(tag="lin", idx=0, B=None, T=None):
    g = np.load(os.path.join(ROOT, "tests", "golden", "ref_sampler.npz"))
    out = {k: g[f"{tag}_{idx}_{k}"] for k in ("u", "seq", "pos", "neg", "timeseq", "hours", "days")}
    if B is not None:
        out = {k: v[:B] for k, v in out.items()}
    if T is not None:
        out = {k: (v[:, -T:] if v.ndim == 2 else v) for k, v in out.items()}
    return out


def oracle_batch(b):
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a))  # noqa: E731
    return {"input_seq": t(b["seq"]), "pos": t(b["pos"]), "neg": t(b["neg"]), "time_seq": t(b["timeseq"]),
            "hours": t(b["hours"]), "days": t(b["days"])}


def dropout_hook(eng, rate):
    """Oracle `drop` callback that asks the library under test for the keep-mask of each site (same seed / step)."""
    def drop(site, x):
        if rate <= 0:
            return x
        n = x.numel()
        keep = torch.empty(n, dtype=torch.uint8, device=eng.device)
        rc = eng.lib.cast_dropout_keep(rate, eng.seed, eng.step_ptr, site, n, keep.data_ptr(), eng._stream())
        assert rc == 0
        k = keep.cpu().to(x.dtype).reshape(x.shape)
        return x * k / (1.0 - rate)
    return drop


def rel_err(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


class WorstErrors:
    """Largest relative error per (backend, kernel, tensor) that a test module has seen; `report` prints them (at the
    module's teardown) past pytest's output capture, so a test log records what the tolerances had to cover."""

    def __init__(self, title):
        self.title, self.worst = title, {}

    def note(self, kind, kernel, what, err, where=""):
        key = (kind, kernel, what)
        if err >= self.worst.get(key, (-1.0, ""))[0]:
            self.worst[key] = (err, where)
        return err

    def report(self, config):
        tr = config.pluginmanager.get_plugin("terminalreporter")
        cm = config.pluginmanager.get_plugin("capturemanager")
        if tr is None or cm is None or not self.worst:
            return
        with cm.global_and_fixture_disabled():
            tr.write_line("")
            for kind in sorted({k[0] for k in self.worst}):
                parts = [f"{kern} {what} {e:.2e}" + (f" ({w})" if w else "")
                         for (kd, kern, what), (e, w) in sorted(self.worst.items()) if kd == kind]
                tr.write_line(f"{self.title} [{kind}] worst relative error vs float64: " + ", ".join(parts))


def synth_batch(B, T, itemnum, seed, mean_len=None, max_bins=200):
    """Seeded synthetic batch in the sampler's layout (left-padded seq/pos/neg + time bins, hours, days) for parity
    runs at BASELINE.json shapes the golden fixtures (T=50, B=16) do not reach: ragged lengths (some shorter than
    T, some full), Zipf item popularity (duplicate ids stress the sparse scatter), the newest event in bin 0."""
    rng = np.random.RandomState(seed)
    mean_len = mean_len or 0.8 * T
    prob = np.arange(1, itemnum + 1, dtype=np.float64) ** -1.0
    cdf = np.cumsum(prob / prob.sum())
    cdf[-1] = 1.0
    seq = np.zeros((B, T), np.int32)
    pos = np.zeros((B, T), np.int32)
    neg = np.zeros((B, T), np.int32)
    lens = np.clip(rng.lognormal(np.log(mean_len) - 0.32, 0.8, B), 2, T + 1).astype(np.int64)
    lens[0] = T + 1      # one full row
    lens[-1] = 2         # one almost empty row
    for b in range(B):
        n = int(lens[b])
        items = np.searchsorted(cdf, rng.rand(n)) + 1
        k = n - 1
        seq[b, T - k:] = items[:-1]
        pos[b, T - k:] = items[1:]
        neg[b, T - k:] = rng.randint(1, itemnum + 1, k)
    live = seq > 0
    ts = np.where(live, np.minimum(max_bins, rng.geometric(0.05, (B, T)) - 1), 0).astype(np.int32)
    ts[:, -1] = 0
    hrs = np.where(live, rng.randint(1, 25, (B, T)), 0).astype(np.int32)
    dys = np.where(live, rng.randint(1, 8, (B, T)), 0).astype(np.int32)
    return {"u": np.arange(1, B + 1, dtype=np.int32), "seq": seq, "pos": pos, "neg": neg, "timeseq": ts,
            "hours": hrs, "days": dys}


KINK_TAU = 2e-5


class relu_kink_hook:
    """Context manager: while active, the oracle takes the ReLU derivative of units whose pre-activation lies within
    KINK_TAU of zero (fp32 noise of the H-term dot products; a handful of units per block at BASELINE sizes) from the
    device buffers of the step that has just run — everywhere else the oracle's own sign stands.  `self.ambiguous`
    counts the overridden units, `self.total` all units seen, so tests can assert the override stays negligible."""

    def __init__(self, eng, c, rate):
        self.eng, self.c, self.rate = eng, c, rate
        self.ambiguous = self.total = 0

    def device_active(self, site):
        c = self.c
        if site == O.SITE_MLP0:
            return (c.mlp_h > 0).cpu(), None
        if site == O.SITE_MLP1:   # cast_9 masks the MLP output afterwards: padded rows read 0 there, which is their
            return (c.mlp_out > 0).cpu(), None   # derivative as well (the mask multiplies the gradient)
        tower = {v: k for k, v in O.TOWER_ID.items()}[site // 1000]
        blk = c.tw[tower].blocks[(site % 1000) // 10]
        act = (blk.h1d > 0).cpu()            # active AND kept by the hidden dropout
        keep = None
        if self.rate > 0:
            eng = self.eng
            n = act.numel()
            k = torch.empty(n, dtype=torch.uint8, device=eng.device)
            rc = eng.lib.cast_dropout_keep(self.rate, eng.seed, eng.step_ptr, site, n, k.data_ptr(), eng._stream())
            assert rc == 0
            keep = k.cpu().bool().reshape(act.shape)
        return act, keep

    def __call__(self, site, pre):
        mask = pre > 0
        amb = pre.abs() < KINK_TAU
        self.total += pre.numel()
        if bool(amb.any()):
            act, keep = self.device_active(site)
            act = act.reshape(pre.shape)
            sel = amb if keep is None else amb & keep.reshape(pre.shape)   # a dropped unit has no gradient anyway
            self.ambiguous += int(sel.sum())
            mask = torch.where(sel, act, mask)
        return mask

    def __enter__(self):
        O.RELU_HOOK = self
        return self

    def __exit__(self, *exc):
        O.RELU_HOOK = None
        return False
