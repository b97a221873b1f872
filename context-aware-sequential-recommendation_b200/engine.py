"""Host-side orchestration of the SASRec / CAST hot path on top of the C ABI (include/cast_b200.h).

PyTorch is used for device memory, streams, CUDA-graph capture and (in `dist.py`) NCCL process groups only; every
arithmetic step of the path is a kernel from `csrc/` reached through ctypes.  The structure mirrors the reference
graph builders (`models/sasrec.py:21-125`, `models/cast_N.py`): embedding stage -> context towers -> merge ->
main tower -> loss -> backward -> TF-Adam.

Parameter names are role based (`item_emb`, `main.0.q.w`, ...); `checkpoint.py` maps them to the reference's
TensorFlow variable names (SURVEY.md Appendix B).
"""
from __future__ import annotations

import ctypes as C
import math
import os
from types import SimpleNamespace
from typing import Dict, List, Optional

import numpy as np
import torch

from . import _lib

TOWER_ID = {"main": 0, "time": 1, "hours": 2, "days": 3}
SITE_EMBED, SITE_CONCAT_A, SITE_CONCAT_B = 9000, 9001, 9002
MODELS = ["cast_1", "cast_2", "cast_3", "cast_4", "cast_5", "cast_6", "cast_7", "cast_8", "cast_9", "sasrec",
          "sasrec_static"]  # reference main.py:28
TABLE_ROWS = {"hours_emb": 25, "days_emb": 8}  # reference cast_3.py:34,45 ("24 hours / 7 days + zero padding")
OPTIMIZERS = ["adam", "lazy_adam"]


def block_site(tower: str, block: int, k: int) -> int:
    return 1000 * TOWER_ID[tower] + 10 * block + k


def sinusoid_table(dim: int, length: int) -> np.ndarray:
    """reference modules.py:27-37: pos / 10000**(2*i/dim) with the raw column index i, sin on even FLAT indices and
    cos on odd ones, evaluated in float64 and cast to float32."""
    pos = np.arange(length, dtype=np.float64)[:, None]
    i = np.arange(dim, dtype=np.float64)[None, :]
    v = (pos / np.power(10000.0, 2.0 * i / dim)).reshape(-1)
    v[::2] = np.sin(v[::2])
    v[1::2] = np.cos(v[1::2])
    return v.reshape(length, dim).astype(np.float32)


def model_plan(model: str, args) -> SimpleNamespace:
    """What a registry name is made of (towers, tables, merge) — reference models/*.py, SURVEY.md §3d."""
    m = model.lower()
    if m not in MODELS:
        raise ValueError(f"provide model from {MODELS}")
    L, Lc = args.num_blocks, getattr(args, "num_context_blocks", 2)
    p = SimpleNamespace(model=m, towers={}, tables=["item_emb"], learned_pos=m in ("sasrec", "cast_9"))
    if m in ("cast_1", "cast_2", "cast_3", "cast_4", "cast_5", "cast_6"):
        p.towers["time"] = L
        p.tables.append("time_emb")
    if m in ("cast_3", "cast_4", "cast_5", "cast_6", "cast_7", "cast_8", "cast_9"):
        p.tables += ["hours_emb", "days_emb"]
    if m == "cast_8":
        p.towers["hours"] = L
        p.towers["days"] = L
    if m == "cast_9":
        p.towers["hours"] = Lc
        p.towers["days"] = Lc
        p.towers["time"] = Lc
        p.tables.append("time_emb")
    p.towers["main"] = L
    # embedding stage of the item stream: (add time stream, dropout, mask)
    p.embed = {"sasrec": (False, True, True), "sasrec_static": (False, True, True), "cast_1": (True, True, True),
               "cast_2": (False, False, True), "cast_3": (True, False, True), "cast_4": (False, False, True),
               "cast_5": (True, False, False), "cast_6": (False, False, False), "cast_7": (False, False, True),
               "cast_8": (False, False, True), "cast_9": (False, False, False)}[m]
    # merge MLP: (sources, width covered by dropout A, second dropout B, position relative to main tower, mask after)
    p.merge = {"cast_2": (["seq", "time"], 2, False, "pre", False),
               "cast_3": (["seq", "hours", "days"], 3, False, "pre", False),
               "cast_4": (["seq", "time", "hours", "days"], 2, True, "pre", False),
               "cast_5": (["seq", "hours", "days"], 3, False, "post", False),
               "cast_6": (["seq", "time", "hours", "days"], 2, True, "post", False),
               "cast_7": (["seq", "hours", "days"], 3, False, "pre", False),
               "cast_8": (["seq", "hours", "days"], 3, False, "pre", False),
               "cast_9": (["seq", "time", "hours", "days"], 4, False, "pre", True)}.get(m)
    # which tower's last-block attention map the reference exposes as `attention_weights`
    p.attn_tower = "time" if m in ("cast_1", "cast_2", "cast_3", "cast_4", "cast_5", "cast_6") else "main"
    return p


def shard_rows(itemnum: int, world: int) -> int:
    """Rows of one rank's shard of the item table (uniform over ranks): cyclic ownership id -> rank id % world, local
    row id // world, +1 on ranks > 0 whose local row 0 is a never-referenced pad (csrc/cast_rt.cuh TableRef)."""
    return (itemnum + 1 + world - 1) // world + 1


def param_shapes(plan, args, itemnum: int, item_rows: Optional[int] = None):
    """Ordered (name, shape, fan_in, fan_out | None) — tables first so the l2_emb region is contiguous.  With a
    row-sharded item table (item_rows = rows of this rank's shard) the first tensor is the local shard; its glorot
    fan-in stays the full vocabulary."""
    H, T = args.hidden_units, args.maxlen
    out = []
    rows = {"item_emb": itemnum + 1, "time_emb": args.max_bins + 1, **TABLE_ROWS}
    for t in plan.tables:
        if t == "item_emb" and item_rows is not None:
            out.append((t, (item_rows, H), rows[t], H))
            continue
        out.append((t, (rows[t], H), rows[t], H))
    if plan.learned_pos:
        out.append(("pos_emb", (T, H), T, H))
    n_tables = len(out)
    for tower, nb in plan.towers.items():
        for i in range(nb):
            pre = f"{tower}.{i}."
            out.append((pre + "ln1.beta", (H,), None, 0.0))
            out.append((pre + "ln1.gamma", (H,), None, 1.0))
            for d in ("q", "k", "v"):
                out.append((pre + d + ".w", (H, H), H, H))
                out.append((pre + d + ".b", (H,), None, 0.0))
            out.append((pre + "ln2.beta", (H,), None, 0.0))
            out.append((pre + "ln2.gamma", (H,), None, 1.0))
            for d in ("ffn1", "ffn2"):
                out.append((pre + d + ".w", (H, H), H, H))
                out.append((pre + d + ".b", (H,), None, 0.0))
        out.append((f"{tower}.lnf.beta", (H,), None, 0.0))
        out.append((f"{tower}.lnf.gamma", (H,), None, 1.0))
    if plan.merge:
        k = len(plan.merge[0]) * H
        out += [("mlp.0.w", (k, k), k, k), ("mlp.0.b", (k,), None, 0.0), ("mlp.1.w", (k, H), k, H),
                ("mlp.1.b", (H,), None, 0.0)]
    return out, n_tables


class Engine:
    """Owns parameters, optimizer state, activations and launches.  One instance per process / GPU."""

    def __init__(self, model: str, usernum: int, itemnum: int, args, device=None, lib=None, seed: Optional[int] = None,
                 item_shard: Optional[tuple] = None, alloc=None, fused: bool = True):
        """item_shard = (rank, world): this process owns one row shard of the item table (BASELINE config 5; the
        other shards are read over NVLink peer mappings once dist.attach has exchanged them).  alloc(numel, dtype) ->
        tensor: allocator for the buffers peers read (CPU tests: POSIX shared memory; default torch).
        fused=False runs every block on the generic LayerNorm + GEMM kernels even where the row kernels apply (the
        reference the row kernels are tested against); widths the row kernels do not take run there too.

        args.optimizer (default "adam"): "adam" is the reference's dense TF-Adam on every parameter.  "lazy_adam" is
        tf.contrib.opt.LazyAdamOptimizer on the item table: a step updates w, m and v of the table rows its batch touches
        (the distinct nonzero ids of seq, pos and neg, over all ranks) with the dense update's arithmetic and bias
        correction, and leaves every other row bit for bit as it was (row 0 and a shard's pad row never move); all other
        parameters keep dense TF-Adam.  The step's table cost then follows the batch instead of the catalog.  It is a
        different optimizer (m and v of a row decay only when the row is touched), so it is opt-in; it refuses
        l2_emb != 0, whose table-wide decay cannot be lazy.

        args.clip_grad (default False): global-norm gradient clipping with the threshold args.max_norm (the reference's
        flag, default 5.0), as tf.clip_by_global_norm over every parameter's gradient as Adam consumes it (divided by
        the global sum(istarget), plus l2_emb * w on the tables; under lazy_adam untouched rows count as 0; under data
        parallelism the rank-ordered sum; with a row-sharded table every shard).  norm = sqrt(sum g^2) in fp64, Adam
        steps on g * scale with scale = max_norm / norm if norm > max_norm else 1 (NaN for a non-finite norm).  The
        norm, the scale and the update run on the device inside the step; a step below the threshold gives the bits of
        clipping off."""
        self.lib = lib if lib is not None else _lib.load_library()
        self.timing = None
        if device is None:
            if not torch.cuda.is_available():
                raise _lib.CastError("no CUDA device: this package has no CPU fallback")
            device = torch.device("cuda", torch.cuda.current_device())
        self.device = torch.device(device)
        self.args = args
        self.plan = model_plan(model, args)
        self.usernum, self.itemnum = usernum, itemnum
        self.H, self.T, self.h = args.hidden_units, args.maxlen, args.num_heads
        if self.H % self.h:
            raise ValueError("hidden_units must be divisible by num_heads")
        self.rate = float(args.dropout_rate)
        self.lr = float(args.lr)
        self.l2 = float(getattr(args, "l2_emb", 0.0))
        self.optimizer = getattr(args, "optimizer", "adam")
        if self.optimizer not in OPTIMIZERS:
            raise ValueError(f"optimizer must be one of {OPTIMIZERS}, got {self.optimizer!r}")
        if self.optimizer == "lazy_adam" and self.l2:
            raise ValueError("optimizer 'lazy_adam' cannot apply l2_emb: a table-wide decay would touch every row")
        self.seed = int(seed if seed is not None else (getattr(args, "seed", 0) or 0))
        self.beta1, self.beta2, self.eps = 0.9, 0.98, 1e-8  # models/sasrec.py:120 (beta2=0.98), TF defaults else
        self.item_shard = tuple(item_shard) if item_shard is not None and item_shard[1] > 1 else None
        self.V_items = itemnum + 1
        self.shard_R = shard_rows(itemnum, self.item_shard[1]) if self.item_shard else None
        # the shard map (local_rows / global_ids): row 0 of ranks > 0 is a pad; item_rows = rows of this process's item
        # table that hold items, counting that pad
        self.shard_pad = 1 if self.item_shard is not None and self.item_shard[0] > 0 else 0
        self.item_rows = self.V_items
        if self.item_shard is not None:
            rank, world = self.item_shard
            self.item_rows = (self.V_items - rank + world - 1) // world + self.shard_pad
        self.alloc = alloc
        self.arena = None
        if self.item_shard is not None and alloc is None:
            from . import dist as _dist      # peer-visible buffers (table shard, sorted entries, source rows)
            self.arena = _dist.PeerArena(self.lib, self.device)
            self.alloc = self.arena.alloc
        shapes, n_tables = param_shapes(self.plan, args, itemnum, self.shard_R)
        self.shapes = shapes
        total = sum(int(np.prod(s)) for _, s, _, _ in shapes)
        f32 = dict(dtype=torch.float32, device=self.device)
        self.w = self._peer_zeros(total, torch.float32)
        self.gbuf = torch.zeros(total + 4, **f32)  # gradients + {loss_sum, auc_sum, count, pad}: one collective
        self.g = self.gbuf[:total]
        self.sums = self.gbuf[total:]
        self.m = torch.zeros(total, **f32)
        self.v = torch.zeros(total, **f32)
        self.P: Dict[str, torch.Tensor] = {}
        self.G: Dict[str, torch.Tensor] = {}
        self.offsets: Dict[str, int] = {}
        off = 0
        for idx, (name, shape, _, _) in enumerate(shapes):
            n = int(np.prod(shape))
            self.P[name] = self.w[off:off + n].view(*shape)
            self.G[name] = self.g[off:off + n].view(*shape)
            self.offsets[name] = off
            off += n
            if idx == n_tables - 1:
                self.l2_hi = off
        self.n_params = total
        self.adam_state = torch.zeros(2, dtype=torch.int64, device=self.device)  # {f32 b1p, f32 b2p, u64 step}
        self.step_ptr = self.adam_state.data_ptr() + 8
        # lazy_adam: the gradient epoch (advanced once per backward pass, never rewound) and each item-table row's stamp
        # = the epoch of the last backward pass that wrote its gradient (csrc/scatter.cu, csrc/adam.cu).  Data
        # parallelism moves both into peer-visible memory (dist.attach).
        self.grad_epoch = self.stamp = None
        self.peer_stamps = None     # set by dist.attach(): device arrays of the ranks' stamp / epoch pointers
        if self.optimizer == "lazy_adam":
            self.grad_epoch = torch.zeros(1, dtype=torch.int32, device=self.device)
            self.stamp = torch.zeros(self.P["item_emb"].shape[0], dtype=torch.int32, device=self.device)
        # clip_grad: fp64 sum-of-squares partials (cast_clip_parts() per pass; a row shard's go to peer-visible memory
        # that the other ranks fold) and the step's {scale, pre-clip norm}
        self.clip = bool(getattr(args, "clip_grad", False))
        self.max_norm = float(getattr(args, "max_norm", 5.0))
        self.clip_out = self.clip_parts = self.clip_shard_parts = None
        self.clip_peers = None      # set by dist.attach_sharded(): (barrier, device array of the ranks' shard partials)
        if self.clip:
            if not (math.isfinite(self.max_norm) and self.max_norm > 0):
                raise ValueError(f"clip_grad needs a finite max_norm > 0, got {self.max_norm}")
            self.clip_nparts = int(self.lib.cast_clip_parts())
            self.clip_parts = torch.zeros(2 * self.clip_nparts, dtype=torch.float64, device=self.device)
            self.clip_out = torch.zeros(2, dtype=torch.float32, device=self.device)
            if self.item_shard is not None:
                self.clip_shard_parts = self._peer_zeros(self.clip_nparts, torch.float64)
        self.sinus = torch.from_numpy(sinusoid_table(self.H, self.T)).to(self.device)
        self.init_parameters(self.seed or 42)
        self._call(self.lib.cast_adam_init_state, self.adam_state.data_ptr(), self.beta1, self.beta2, self._stream())
        self._ctx: Dict[int, SimpleNamespace] = {}
        # The kernels every transformer block runs on, fixed for the engine's lifetime: with row_kernels the forward
        # runs on the tcgen05 row kernels (csrc/row_umma.cu, cast_rowk_supported(H)), the backward on the mma.sync row
        # kernels (csrc/fused.cu), and the gradient partial sums wait for one reduction launch per step; otherwise
        # LayerNorm kernels + cast_gemm / cast_colsum.
        self.row_kernels = bool(fused and self.lib.cast_rowk_supported(self.H))
        names = [f"{tower}.{i}." for tower, nb in self.plan.towers.items() for i in range(nb)]
        # per-block weight operand images, rebuilt once per forward pass (cast_rowk_presplit); none without blocks
        self.rowk_img = None
        if self.row_kernels and names:
            self.rowk_block = {n: j for j, n in enumerate(names)}
            self.rowk_img_bytes = int(self.lib.cast_rowk_image_bytes(self.H))
            self.rowk_img = torch.zeros(len(names) * self.rowk_img_bytes, dtype=torch.uint8, device=self.device)
            ptrs = [self.P[n + w].data_ptr() for n in names for w in ("q.w", "k.w", "v.w", "ffn1.w", "ffn2.w")]
            self.rowk_wptrs = (C.c_void_p * len(ptrs))(*ptrs)
        # final LayerNorm + loss + LayerNorm backward in one launch: the main tower's output must be seq_emb itself
        self.fuse_tail = (self.row_kernels and self.item_shard is None
                          and not (self.plan.merge and self.plan.merge[3] == "post"))
        self.world_size = 1
        self.grad_allreduce = None  # set by dist.attach(); called between backward and Adam
        self.adam_g = self.gbuf     # what Adam consumes: the local buffer, or the rank-ordered sum (dist.PeerExchange)
        self.exchange_capturable = False   # dist.attach*: the exchange is plain kernel launches (the step is one graph)
        self.after_adam = None      # set by dist.attach_sharded(): the barrier that ends a row-sharded step
        # the step's kernels form a chain whose operands obey include/cast_b200.h's cast_set_pdl contract (weights are
        # last written by the optimizer pass of the previous step, images on a joined side stream, activations of the
        # forward pass long before the backward kernels that re-read them): programmatic dependent launch is safe here
        if self.device.type == "cuda":
            self.lib.cast_set_pdl(0 if os.environ.get("CAST_PDL", "1") == "0" else 1)
        self.before_backward = None  # set by dist.attach(): the barrier that lets this step overwrite the gradient buffer
        self.peer_adam = None       # set by dist.attach(): (device pointer table, n_ranks, g_red) => Adam sums the ranks' buffers
        self.shard_ptrs = None      # ... device array of the ranks' item-table shard pointers (own + peer mappings)

    # ------------------------------------------------------------------ plumbing
    def _peer_zeros(self, numel, dtype):
        """a buffer other ranks may read (item-table shard, sorted gradient entries, their source rows)"""
        if self.alloc is not None and self.item_shard is not None:
            t = self.alloc(int(numel), dtype)
            t.zero_()
            return t
        return torch.zeros(int(numel), dtype=dtype, device=self.device)

    def _stream(self):
        if self.device.type == "cuda":
            return torch.cuda.current_stream(self.device).cuda_stream
        return None

    def _call(self, fn, *a):
        if self.timing is not None:  # per-call CUDA events on the launch stream (bench / profiling only)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            rc = fn(*a)
            e1.record()
            self.timing.append((fn.__name__, a, e0, e1))
        else:
            rc = fn(*a)
        if rc != 0:
            _lib.check(self.lib, rc, fn.__name__)

    def _fork(self, c, name: str, fn) -> bool:
        """Runs fn() on the context's side stream `name` after the work enqueued so far on the current stream: a
        parallel branch of the step (and of its captured graph) until _join(c, name).  Where the step runs in stream
        order (no CUDA device, per-call timing) nothing is enqueued and it returns False."""
        if self.device.type != "cuda" or self.timing is not None:
            return False
        s = c.streams.get(name)
        if s is None:
            s = c.streams[name] = torch.cuda.Stream(device=self.device)
        s.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(s):
            fn()
        c.forked[name] = s
        return True

    def _join(self, c, name: str) -> bool:
        """The current stream waits for the branch `name` if it is forked; returns whether it was."""
        s = c.forked.pop(name, None)
        if s is None:
            return False
        torch.cuda.current_stream(self.device).wait_stream(s)
        return True

    @staticmethod
    def _p(t):
        return None if t is None else t.data_ptr()

    def init_parameters(self, seed: int):
        """TF-1.15 default initialisers (SURVEY A-17): glorot-uniform for tables and kernels, zeros for biases and
        beta, ones for gamma.  (The draws are this repo's: TF's graph-level seeding is not reproducible.)"""
        gen = torch.Generator().manual_seed(seed)
        for name, shape, fan_in, fan_out in self.shapes:
            if fan_in is None:
                self.P[name].fill_(float(fan_out))
            else:
                limit = math.sqrt(6.0 / (fan_in + fan_out))
                if name == "item_emb" and self.item_shard is not None:
                    # the same draws as the unsharded table, then this rank's rows
                    full = (torch.rand((self.V_items, shape[1]), generator=gen, dtype=torch.float64) * 2 - 1)
                    self.P[name].copy_(self.shard_of(full.mul(limit).float()).to(self.device))
                    continue
                vals = (torch.rand(shape, generator=gen, dtype=torch.float64) * 2 - 1).mul(limit).float()
                self.P[name].copy_(vals.to(self.device))
        self.m.zero_()
        self.v.zero_()

    def shard_of(self, full: torch.Tensor) -> torch.Tensor:
        """rows of the full [V, H] item table (or of any per-item tensor) that live in this rank's shard, in local order"""
        rank, world = self.item_shard
        out = torch.zeros((self.shard_R,) + tuple(full.shape[1:]), dtype=full.dtype)
        mine = full[rank::world]
        out[self.shard_pad:self.shard_pad + mine.shape[0]] = mine
        return out

    def local_rows(self, ids: np.ndarray) -> np.ndarray:
        """global item ids -> rows of this process's item table, 0 where the id is not on this shard (the identity
        without a row-sharded table).  The map is increasing on the ids a shard holds."""
        if self.item_shard is None:
            return ids
        rank, world = self.item_shard
        mine = (ids % world == rank) & (ids > 0) & (ids < self.V_items)
        return np.where(mine, ids // world + self.shard_pad, 0)

    def global_ids(self, rows: torch.Tensor) -> torch.Tensor:
        """rows of this process's item table -> global item ids, row 0 -> 0 (the inverse of local_rows; the identity
        without a row-sharded table)"""
        if self.item_shard is None:
            return rows
        rank, world = self.item_shard
        return torch.where(rows > 0, (rows - self.shard_pad) * world + rank, rows)

    def rebind_gradients(self, gbuf: torch.Tensor):
        """move the flat gradient buffer (and every view of it) to `gbuf` — peer-visible memory for data parallelism"""
        assert gbuf.numel() == self.gbuf.numel()
        local = self.adam_g is self.gbuf
        self.gbuf = gbuf
        self.g = gbuf[:self.n_params]
        self.sums = gbuf[self.n_params:]
        for name, shape, _, _ in self.shapes:
            off = self.offsets[name]
            self.G[name] = self.g[off:off + int(np.prod(shape))].view(*shape)
        if local:
            self.adam_g = gbuf
        for c in self._ctx.values():
            c.sums = self.sums

    def global_sums(self) -> torch.Tensor:
        """{sum loss terms, sum auc terms, sum istarget, pad} of the whole (global) batch after the exchange"""
        return self.adam_g[self.n_params:]

    def load_parameters(self, params: Dict[str, "torch.Tensor | np.ndarray"]):
        for k, v in params.items():
            v = torch.as_tensor(np.asarray(v) if not torch.is_tensor(v) else v)
            if k == "item_emb" and self.item_shard is not None and v.shape[0] == self.V_items:
                v = self.shard_of(v)
            self.P[k].copy_(v.to(self.device))

    def state_step(self) -> int:
        return int(self.adam_state[1].item())

    # ------------------------------------------------------------------ buffers
    def ctx(self, B: int) -> SimpleNamespace:
        c = self._ctx.get(B)
        if c is not None:
            return c
        H, T, h, dev = self.H, self.T, self.h, self.device
        N = B * T
        lib = self.lib
        f = lambda *s: torch.empty(*s, dtype=torch.float32, device=dev)  # noqa: E731
        # buffers the other ranks read during the row-sharded gradient exchange (dist.attach_sharded)
        fp = (lambda *s: self._peer_zeros(int(np.prod(s)), torch.float32).view(*s)) if self.item_shard else f
        c = SimpleNamespace(B=B, N=N)
        c.streams = {}       # name -> side stream of this context (_fork), created on first use
        # per step, left empty by launch_fwd_bwd: the side-stream branches forked and not yet joined (name -> stream)
        # and the deferred gradient partial sums (flush_reduce_jobs)
        c.forked = {}
        c.reduce_jobs = []
        c.keys3 = torch.zeros(3, N, dtype=torch.int32, device=dev)   # input_seq | pos | neg
        c.cids = torch.zeros(3, N, dtype=torch.int32, device=dev)    # time_seq | hours | days
        c.tw = {}
        for tower, nb in self.plan.towers.items():
            blocks = []
            for _ in range(nb):
                b = SimpleNamespace()
                for nm in ("qn", "Q", "K", "V", "y", "zn", "h1d", "xout"):
                    setattr(b, nm, f(N, H))
                for nm in ("mu1", "rs1", "kmask", "qmask", "mu2", "rs2"):
                    setattr(b, nm, f(N))
                for nm in ("rmax", "rlinv", "rowD"):
                    setattr(b, nm, f(B * h * T))
                if self.row_kernels:
                    # own partial buffers per block: the fixed-order reduction of all blocks is one launch at the end
                    # of backward (cast_reduce_partials_batch) instead of one small launch per fused backward kernel
                    nws = self.lib.cast_block_bwd_workspace_bytes(N, H) // 4 + 16
                    b.ws_ffn, b.ws_qkv = f(nws), f(nws)
                blocks.append(b)
            # x_last: the main tower's last block output, normalised by cast_lnf_loss (fuse_tail);
            # ws_lnf: the gamma/beta partials of the final LayerNorm's backward (row-kernel paths, unless fuse_tail)
            lnf_partials = self.row_kernels and not (tower == "main" and self.fuse_tail)
            c.tw[tower] = SimpleNamespace(blocks=blocks, out=(fp if tower == "main" else f)(N, H), muf=f(N), rsf=f(N),
                                          dx_in=f(N, H), x_in=None, x_last=None,
                                          ws_lnf=f(lib.cast_layernorm_bwd_workspace_bytes(N, H) // 4 + 16)
                                          if lnf_partials else None)
        # attention backward scratch: P~ and dS of one block ([2][h*B,T,T]), shared by all blocks (d <= 64 only)
        c.attn_ws = None
        if H // h <= 64 and 2 * B * h * T * T * 4 <= (2 << 30):
            c.attn_ws = torch.empty(self.lib.cast_attn_bwd_workspace_bytes(B, T, h) // 4, dtype=torch.float32, device=dev)
        c.x0 = f(N, H)
        c.emb = {t: f(N, H) for t in self.plan.tables if t != "item_emb"}
        c.demb = {t: f(N, H) for t in self.plan.tables if t != "item_emb"}
        if self.plan.merge:
            k = len(self.plan.merge[0])
            c.cat, c.mlp_h, c.mlp_out = f(N, k * H), f(N, k * H), fp(N, H)
            c.dcat, c.dmlp_h, c.dmlp_o = f(N, k * H), f(N, k * H), f(N, H)
            c.dsrc = {s: f(N, H) for s in self.plan.merge[0]}
        c.pos_logits, c.neg_logits, c.gpos, c.gneg = f(N), f(N), fp(N), fp(N)
        c.sums = self.sums  # loss_sum, auc_sum, count (tail of the gradient buffer)
        c.dseq = f(N, H)
        c.t = [f(N, H) for _ in range(7)]  # gradient scratch
        c.g0 = fp(N, H)
        kmax = (len(self.plan.merge[0]) if self.plan.merge else 1) * H
        c.splits = int(max(1, min(296, N // 128)))
        ws = max(lib.cast_layernorm_bwd_workspace_bytes(N, H),
                 lib.cast_gemm_workspace_bytes(kmax, kmax, N, c.splits), lib.cast_gemm_workspace_bytes(N, kmax, kmax, 1),
                 lib.cast_colsum_workspace_bytes(N, kmax), lib.cast_colsum_workspace_bytes(B, T * H),
                 lib.cast_logits_loss_workspace_bytes(N), lib.cast_block_bwd_workspace_bytes(N, H))
        c.ws = torch.empty(ws // 4 + 16, dtype=torch.float32, device=dev)
        c.ws_bytes = ws
        # the training step's loss partial sums, reduced with the other deferred jobs: cast_lnf_loss's (fuse_tail,
        # with the final LayerNorm's gamma/beta partials) or cast_logits_loss's
        c.ws_tail = f(lib.cast_lnf_loss_workspace_bytes(N, H) // 4 + 16) if self.fuse_tail else None
        c.ws_loss = None if self.fuse_tail else f(lib.cast_logits_loss_workspace_bytes(N) // 4 + 16)
        c.seq_emb = None     # the forward pass's output (forward)
        c.shard_src = None   # the item-table gradient's source rows for the sharded exchange (scatter)
        vmax = max(self.P[t].shape[0] for t in self.plan.tables)
        if self.item_shard:
            vmax = max(vmax, self.item_shard[1] * self.shard_R)   # owner-major key range of the sharded sort
        sws = lib.cast_scatter_workspace_bytes(N, 3, vmax)
        c.sws = self._peer_zeros(sws // 4 + 16, torch.int32) if self.item_shard else \
            torch.empty(sws // 4 + 16, dtype=torch.int32, device=dev)
        c.sws_bytes = sws
        c.peer = None   # pointers into the other ranks' buffers, exchanged on the first sharded step
        spb = lib.cast_scatter_partial_bytes(N, 3, H)
        c.spart = torch.empty(spb // 4 + 16, dtype=torch.float32, device=dev)
        c.spart_bytes = spb
        c.attn = None
        c.graph = None
        self._ctx[B] = c
        return c

    # ------------------------------------------------------------------ op wrappers
    def _gemm(self, A, sam, sak, Bm, sbk, sbn, Cm, ldc, M, N, K, c, bias=None, relu=0, rate=0.0, site=0, act=None,
              ld_act=0, act_scale=1.0, resid=None, ldr=0, row_ids=None, splits=1):
        self._call(self.lib.cast_gemm, A.data_ptr(), sam, sak, Bm.data_ptr(), sbk, sbn, Cm.data_ptr(), ldc, M, N, K,
                   self._p(bias), relu, rate, self.seed, self.step_ptr, site, self._p(act), ld_act, act_scale,
                   self._p(resid), ldr, self._p(row_ids), splits, c.ws.data_ptr(), c.ws_bytes, self._stream())

    def linear_fwd(self, c, X, W, b, Y, **kw):
        N, K = X.shape
        M = W.shape[1]
        self._gemm(X, K, 1, W, M, 1, Y, M, N, M, K, c, bias=b, **kw)

    def linear_dgrad(self, c, dY, W, dX, **kw):
        N, M = dY.shape
        K = W.shape[0]
        self._gemm(dY, M, 1, W, 1, M, dX, K, N, K, M, c, **kw)

    def linear_wgrad(self, c, X, dY, dW, db):
        N, K = X.shape
        M = dY.shape[1]
        self._gemm(X, 1, K, dY, M, 1, dW, M, K, M, N, c, splits=c.splits)
        if db is not None:
            self._call(self.lib.cast_colsum, dY.data_ptr(), N, M, M, db.data_ptr(), c.ws.data_ptr(), c.ws_bytes,
                       self._stream())

    def ln_fwd(self, x, pre, y, mu, rs, xnz=None, ynz=None):
        N = x.shape[0]
        self._call(self.lib.cast_layernorm_fwd, x.data_ptr(), self.P[pre + ".gamma"].data_ptr(),
                   self.P[pre + ".beta"].data_ptr(), N, self.H, 1e-8, y.data_ptr(), self._p(mu), self._p(rs),
                   self._p(xnz), self._p(ynz), self._stream())

    def ln_bwd(self, c, dy, x, mu, rs, pre, dx, dx_add=None):
        N = x.shape[0]
        self._call(self.lib.cast_layernorm_bwd, dy.data_ptr(), x.data_ptr(), mu.data_ptr(), rs.data_ptr(),
                   self.P[pre + ".gamma"].data_ptr(), N, self.H, self._p(dx_add), dx.data_ptr(),
                   self.G[pre + ".gamma"].data_ptr(), self.G[pre + ".beta"].data_ptr(), c.ws.data_ptr(), c.ws_bytes,
                   self._stream())

    def embed_fwd(self, ids, table, out, pos=None, add=None, rate=0.0, site=0, mask_ids=None):
        N = ids.numel()
        if self.item_shard is not None and table is self.P["item_emb"]:
            self._call(self.lib.cast_embed_fwd_sharded, ids.data_ptr(), self.shard_ptrs.data_ptr(), self.item_shard[1],
                       self.V_items, self.H, N, self.T, float(self.H ** 0.5), self._p(pos), self._p(add), rate,
                       self.seed, self.step_ptr, site, self._p(mask_ids), out.data_ptr(), self._stream())
            return
        self._call(self.lib.cast_embed_fwd, ids.data_ptr(), table.data_ptr(), table.shape[0], self.H, N, self.T,
                   float(self.H ** 0.5), self._p(pos), self._p(add), rate, self.seed, self.step_ptr, site,
                   self._p(mask_ids), out.data_ptr(), self._stream())

    def mask_dropout(self, x, ids, rate, site, out_m, out_md):
        N = x.shape[0]
        self._call(self.lib.cast_mask_dropout, x.data_ptr(), self._p(ids), rate, self.seed, self.step_ptr, site, N,
                   x.shape[1], self._p(out_m), self._p(out_md), self._stream())

    def scatter(self, c, keys, nsrc, rows, rowscale, scale, table_name):
        N = c.N
        V = self.P[table_name].shape[0]
        rows_a = (C.c_void_p * nsrc)(*[r.data_ptr() for r in rows])
        rs_a = (C.c_void_p * nsrc)(*[(r.data_ptr() if r is not None else None) for r in rowscale])
        sc_a = (C.c_float * nsrc)(*scale)
        if table_name == "item_emb" and self.item_shard is not None:
            if not self._join(c, "sort"):   # sorted on a side stream during the forward pass (launch_fwd_bwd)
                self._call(self.lib.cast_scatter_sort_sharded, keys.data_ptr(), nsrc, N, self.V_items,
                           self.item_shard[1], self.shard_R, c.sws.data_ptr(), c.sws_bytes, self._stream())
            if rows[0] is not c.g0:    # peers read the input-sequence gradient from the exported buffer
                c.g0.copy_(rows[0])
            c.shard_src = (nsrc, [c.g0] + list(rows[1:]), list(rowscale), list(scale))
            return
        if table_name == "item_emb" and self.stamp is not None:   # lazy: no zeroing pass, touched rows get stamped
            if not self._join(c, "sort"):
                self._call(self.lib.cast_scatter_sort, keys.data_ptr(), nsrc, N, V, c.sws.data_ptr(), c.sws_bytes,
                           self._stream())
            self._call(self.lib.cast_scatter_apply_lazy, nsrc, N, rows_a, rs_a, sc_a, V, self.H,
                       self.G[table_name].data_ptr(), c.sws.data_ptr(), c.sws_bytes, c.spart.data_ptr(),
                       c.spart_bytes, self.stamp.data_ptr(), self.grad_epoch.data_ptr(), self._stream())
            return
        if table_name == "item_emb" and self._join(c, "sort"):   # the ids are sorted already: only the sums remain
            self._call(self.lib.cast_scatter_apply, nsrc, N, rows_a, rs_a, sc_a, V, self.H,
                       self.G[table_name].data_ptr(), c.sws.data_ptr(), c.sws_bytes, c.spart.data_ptr(),
                       c.spart_bytes, 0, self._stream())
            return
        self._call(self.lib.cast_scatter_rows, keys.data_ptr(), nsrc, N, rows_a, rs_a, sc_a, V, self.H,
                   self.G[table_name].data_ptr(), c.sws.data_ptr(), c.sws_bytes, c.spart.data_ptr(), c.spart_bytes,
                   self._stream())

    # ------------------------------------------------------------------ towers
    def tower_fwd(self, c, tower, x_in, ids, train, want_attn=False):
        """L x (LN, MHA, LN, FFN, *= mask) + final LN — reference models/sasrec.py:65-85."""
        tb = c.tw[tower]
        tb.x_in = x_in
        rate = self.rate if train else 0.0
        H, B, T, h = self.H, c.B, self.T, self.h
        x = x_in
        nb = len(tb.blocks)
        self._join(c, "presplit")   # the rowk weight split, if launch_fwd_bwd forked it
        P = self.P
        for i, b in enumerate(tb.blocks):
            pre = f"{tower}.{i}."
            if self.row_kernels:
                self._call(self.lib.cast_rowk_ln_qkv_fwd, x.data_ptr(), P[pre + "ln1.gamma"].data_ptr(),
                           P[pre + "ln1.beta"].data_ptr(), P[pre + "q.b"].data_ptr(), P[pre + "k.b"].data_ptr(),
                           P[pre + "v.b"].data_ptr(), self.rowk_image(pre), c.N, H, 1e-8, b.qn.data_ptr(),
                           b.Q.data_ptr(), b.K.data_ptr(), b.V.data_ptr(), b.mu1.data_ptr(), b.rs1.data_ptr(),
                           b.kmask.data_ptr(), b.qmask.data_ptr(), self._stream())
            else:
                self.ln_fwd(x, pre + "ln1", b.qn, b.mu1, b.rs1, b.kmask, b.qmask)
                self.linear_fwd(c, b.qn, self.P[pre + "q.w"], self.P[pre + "q.b"], b.Q)
                self.linear_fwd(c, x, self.P[pre + "k.w"], self.P[pre + "k.b"], b.K)
                self.linear_fwd(c, x, self.P[pre + "v.w"], self.P[pre + "v.b"], b.V)
            attn = None
            if want_attn and i == nb - 1:
                if c.attn is None or c.attn.shape[0] != h * B:
                    c.attn = torch.empty(h * B, T, T, dtype=torch.float32, device=self.device)
                attn = c.attn
            self._call(self.lib.cast_attn_fwd, b.Q.data_ptr(), H, b.K.data_ptr(), H, b.V.data_ptr(), H,
                       b.qn.data_ptr(), b.kmask.data_ptr(), b.qmask.data_ptr(), B, T, H, h, rate, self.seed,
                       self.step_ptr, block_site(tower, i, 1), ids.data_ptr(), b.y.data_ptr(), self._p(attn),
                       b.rmax.data_ptr(), b.rlinv.data_ptr(), self._stream())
            if self.row_kernels:
                self._call(self.lib.cast_rowk_ln_ffn_fwd, b.y.data_ptr(), P[pre + "ln2.gamma"].data_ptr(),
                           P[pre + "ln2.beta"].data_ptr(), P[pre + "ffn1.b"].data_ptr(), P[pre + "ffn2.b"].data_ptr(),
                           self.rowk_image(pre), ids.data_ptr(), rate, self.seed, self.step_ptr,
                           block_site(tower, i, 2), block_site(tower, i, 3), c.N, H, 1e-8, b.zn.data_ptr(),
                           b.h1d.data_ptr(), b.xout.data_ptr(), b.mu2.data_ptr(), b.rs2.data_ptr(), self._stream())
            else:
                self.ln_fwd(b.y, pre + "ln2", b.zn, b.mu2, b.rs2)
                self.linear_fwd(c, b.zn, self.P[pre + "ffn1.w"], self.P[pre + "ffn1.b"], b.h1d, relu=1, rate=rate,
                                site=block_site(tower, i, 2))
                self.linear_fwd(c, b.h1d, self.P[pre + "ffn2.w"], self.P[pre + "ffn2.b"], b.xout, rate=rate,
                                site=block_site(tower, i, 3), resid=b.zn, ldr=H, row_ids=ids)
            x = b.xout
        if tower == "main" and train and self.fuse_tail:
            tb.x_last = x       # cast_lnf_loss normalises it (and writes tb.out) together with the loss
            return tb.out
        self.ln_fwd(x, tower + ".lnf", tb.out, tb.muf, tb.rsf)
        return tb.out

    def tower_bwd(self, c, tower, d_out, ids, embed_fx=None):
        """Backward of tower_fwd; parameter gradients land in self.G, returns d(loss)/d(x_in) (tb.dx_in).
        embed_fx = (mask ids or None, dropout rate, site, out): on the row-kernel path block 0's kernel also applies the
        backward of `dropout(emb) * mask` (sasrec.py:58-62) and writes the result to `out` (returned instead)."""
        tb = c.tw[tower]
        H, B, T, h = self.H, c.B, self.T, self.h
        rate = self.rate
        scale = 1.0 / (1.0 - rate) if rate > 0 else 1.0
        t = c.t
        nb = len(tb.blocks)
        x_last = tb.blocks[-1].xout if nb else tb.x_in
        dx = t[0]
        if tower == "main" and self.fuse_tail:
            pass                # dx (= t[0]) and the gamma/beta partials were produced by cast_lnf_loss
        elif self.row_kernels:  # final LayerNorm's gamma/beta partials join the step's single reduction launch
            self._call(self.lib.cast_layernorm_bwd, d_out.data_ptr(), x_last.data_ptr(), tb.muf.data_ptr(),
                       tb.rsf.data_ptr(), self.P[tower + ".lnf.gamma"].data_ptr(), c.N, H, None, dx.data_ptr(), None,
                       None, tb.ws_lnf.data_ptr(), tb.ws_lnf.numel() * 4, self._stream())
            parts = self.lib.cast_layernorm_bwd_parts(c.N)
            c.reduce_jobs.append((tb.ws_lnf.data_ptr(), parts, H, self.G[tower + ".lnf.gamma"], 2 * H))
            c.reduce_jobs.append((tb.ws_lnf.data_ptr() + 4 * H, parts, H, self.G[tower + ".lnf.beta"], 2 * H))
        else:
            self.ln_bwd(c, d_out, x_last, tb.muf, tb.rsf, tower + ".lnf", dx)
        P = self.P
        for i in reversed(range(nb)):
            b = tb.blocks[i]
            pre = f"{tower}.{i}."
            x_i = tb.blocks[i - 1].xout if i > 0 else tb.x_in
            gm, gmd, dh, dzn, dy = t[1], t[2], t[3], t[4], t[5]
            # x_out = (dropout(h1d W2 + b2) + zn) * mask                      modules.py:304-311, sasrec.py:83
            if self.row_kernels:
                self._call(self.lib.cast_ffn_bwd, dx.data_ptr(), ids.data_ptr(), b.zn.data_ptr(), b.h1d.data_ptr(),
                           b.y.data_ptr(), b.mu2.data_ptr(), b.rs2.data_ptr(), P[pre + "ln2.gamma"].data_ptr(),
                           P[pre + "ffn1.w"].data_ptr(), P[pre + "ffn2.w"].data_ptr(), rate, self.seed, self.step_ptr,
                           block_site(tower, i, 3), c.N, H, dy.data_ptr(), None,
                           b.ws_ffn.data_ptr(), b.ws_ffn.numel() * 4, self._stream())
                cnt = 2 * H + 2 * (H * H + H)
                c.reduce_jobs.append((b.ws_ffn.data_ptr(), self.lib.cast_block_bwd_parts(c.N, 0), cnt,
                                      self.G[pre + "ln2.beta"], cnt))
            else:
                self.mask_dropout(dx, ids, rate, block_site(tower, i, 3), gm, gmd)
                self.linear_wgrad(c, b.h1d, gmd, self.G[pre + "ffn2.w"], self.G[pre + "ffn2.b"])
                self.linear_dgrad(c, gmd, self.P[pre + "ffn2.w"], dh, act=b.h1d, ld_act=H, act_scale=scale)
                self.linear_wgrad(c, b.zn, dh, self.G[pre + "ffn1.w"], self.G[pre + "ffn1.b"])
                self.linear_dgrad(c, dh, self.P[pre + "ffn1.w"], dzn, resid=gm, ldr=H)
                self.ln_bwd(c, dzn, b.y, b.mu2, b.rs2, pre + "ln2", dy)
            # y = attention(Q, K, V) + qn                                      modules.py:262-269
            dQ, dK, dV = t[1], t[2], t[3]
            self._call(self.lib.cast_attn_bwd, b.Q.data_ptr(), H, b.K.data_ptr(), H, b.V.data_ptr(), H,
                       dy.data_ptr(), b.kmask.data_ptr(), b.qmask.data_ptr(), b.rmax.data_ptr(), b.rlinv.data_ptr(),
                       ids.data_ptr(), b.rowD.data_ptr(), B, T, H, h, rate, self.seed, self.step_ptr,
                       block_site(tower, i, 1),
                       dQ.data_ptr(), H, dK.data_ptr(), H, dV.data_ptr(), H, b.y.data_ptr(), b.qn.data_ptr(),
                       self._p(c.attn_ws), c.attn_ws.numel() * 4 if c.attn_ws is not None else 0, self._stream())
            if self.row_kernels:
                dst = tb.dx_in if i == 0 else t[0]
                if i == 0 and embed_fx is not None:
                    fx_ids, fx_rate, fx_site, dst = embed_fx
                    self._call(self.lib.cast_qkv_bwd_embed, dQ.data_ptr(), dK.data_ptr(), dV.data_ptr(),
                               dy.data_ptr(), x_i.data_ptr(), b.qn.data_ptr(), b.mu1.data_ptr(), b.rs1.data_ptr(),
                               P[pre + "ln1.gamma"].data_ptr(), P[pre + "q.w"].data_ptr(), P[pre + "k.w"].data_ptr(),
                               P[pre + "v.w"].data_ptr(), c.N, H, self._p(fx_ids), float(fx_rate), self.seed,
                               self.step_ptr, int(fx_site), dst.data_ptr(), None, b.ws_qkv.data_ptr(),
                               b.ws_qkv.numel() * 4, self._stream())
                else:
                    self._call(self.lib.cast_qkv_bwd, dQ.data_ptr(), dK.data_ptr(), dV.data_ptr(), dy.data_ptr(),
                               x_i.data_ptr(), b.qn.data_ptr(), b.mu1.data_ptr(), b.rs1.data_ptr(),
                               P[pre + "ln1.gamma"].data_ptr(), P[pre + "q.w"].data_ptr(), P[pre + "k.w"].data_ptr(),
                               P[pre + "v.w"].data_ptr(), c.N, H, dst.data_ptr(), None,
                               b.ws_qkv.data_ptr(), b.ws_qkv.numel() * 4, self._stream())
                cnt = 2 * H + 3 * (H * H + H)
                c.reduce_jobs.append((b.ws_qkv.data_ptr(), self.lib.cast_block_bwd_parts(c.N, 1), cnt,
                                      self.G[pre + "ln1.beta"], cnt))
                dx = dst
                continue
            self.linear_wgrad(c, b.qn, dQ, self.G[pre + "q.w"], self.G[pre + "q.b"])
            self.linear_wgrad(c, x_i, dK, self.G[pre + "k.w"], self.G[pre + "k.b"])
            self.linear_wgrad(c, x_i, dV, self.G[pre + "v.w"], self.G[pre + "v.b"])
            dqn, dxk, dxkv = t[4], t[6], t[0]
            self.linear_dgrad(c, dQ, self.P[pre + "q.w"], dqn, resid=dy, ldr=H)
            self.linear_dgrad(c, dK, self.P[pre + "k.w"], dxk)
            self.linear_dgrad(c, dV, self.P[pre + "v.w"], dxkv, resid=dxk, ldr=H)
            dst = tb.dx_in if i == 0 else t[5]
            self.ln_bwd(c, dqn, x_i, b.mu1, b.rs1, pre + "ln1", dst, dx_add=dxkv)
            dx = dst
        if nb == 0:
            tb.dx_in.copy_(dx)
        return tb.dx_in

    # ------------------------------------------------------------------ merge MLP (modules.py:321-335)
    def merge_fwd(self, c, srcs: Dict[str, torch.Tensor], ids, train):
        names, wa, second, _, mask_after = self.plan.merge
        k = len(names)
        rate = self.rate if train else 0.0
        ptrs = (C.c_void_p * k)(*[srcs[n].data_ptr() for n in names])
        if second:
            ra, sa, rb, sb = rate, SITE_CONCAT_A, rate, SITE_CONCAT_B
        else:  # one dropout over the whole concat: expressed as dropout B with site A
            wa, ra, sa, rb, sb = 0, 0.0, SITE_CONCAT_A, rate, SITE_CONCAT_A
        self._call(self.lib.cast_concat_dropout_fwd, ptrs, k, wa, c.N, self.H, ra, sa, rb, sb, self.seed,
                   self.step_ptr, c.cat.data_ptr(), self._stream())
        self.linear_fwd(c, c.cat, self.P["mlp.0.w"], self.P["mlp.0.b"], c.mlp_h, relu=1)
        self.linear_fwd(c, c.mlp_h, self.P["mlp.1.w"], self.P["mlp.1.b"], c.mlp_out, relu=1,
                        row_ids=ids if mask_after else None)
        return c.mlp_out

    def merge_bwd(self, c, d_out):
        names, wa, second, _, _ = self.plan.merge
        k = len(names)
        rate = self.rate
        n1 = c.N * self.H
        self._call(self.lib.cast_relu_bwd, d_out.data_ptr(), c.mlp_out.data_ptr(), 1.0, c.dmlp_o.data_ptr(), n1,
                   self._stream())
        self.linear_wgrad(c, c.mlp_h, c.dmlp_o, self.G["mlp.1.w"], self.G["mlp.1.b"])
        self.linear_dgrad(c, c.dmlp_o, self.P["mlp.1.w"], c.dmlp_h, act=c.mlp_h, ld_act=k * self.H, act_scale=1.0)
        self.linear_wgrad(c, c.cat, c.dmlp_h, self.G["mlp.0.w"], self.G["mlp.0.b"])
        self.linear_dgrad(c, c.dmlp_h, self.P["mlp.0.w"], c.dcat)
        ptrs = (C.c_void_p * k)(*[c.dsrc[n].data_ptr() for n in names])
        if second:
            ra, sa, rb, sb = rate, SITE_CONCAT_A, rate, SITE_CONCAT_B
        else:
            wa, ra, sa, rb, sb = 0, 0.0, SITE_CONCAT_A, rate, SITE_CONCAT_A
        self._call(self.lib.cast_concat_dropout_bwd, c.dcat.data_ptr(), k, wa, c.N, self.H, ra, sa, rb, sb, self.seed,
                   self.step_ptr, ptrs, self._stream())
        return c.dsrc

    # ------------------------------------------------------------------ whole model
    def rowk_presplit(self, stream):
        self._call(self.lib.cast_rowk_presplit, self.rowk_wptrs, len(self.rowk_block), self.H,
                   self.rowk_img.data_ptr(), self.rowk_img.numel(), stream)

    def rowk_image(self, pre: str) -> int:
        return self.rowk_img.data_ptr() + self.rowk_block[pre] * self.rowk_img_bytes

    def forward(self, c, train: bool, want_attn: bool = False):
        """Builds seq_emb [N,H] from the ids already resident in c.keys3 / c.cids; returns the buffer."""
        plan = self.plan
        ids = c.keys3[0]
        if self.rowk_img is not None and "presplit" not in c.forked:
            self.rowk_presplit(self._stream())   # weights moved since the last step: refresh the operand images
        streams: Dict[str, torch.Tensor] = {}
        for j, (tname, key) in enumerate((("time_emb", "time"), ("hours_emb", "hours"), ("days_emb", "days"))):
            if tname in plan.tables:
                self.embed_fwd(c.cids[j], self.P[tname], c.emb[tname])
                s = c.emb[tname]
                if key in plan.towers:
                    s = self.tower_fwd(c, key, s, ids, train, want_attn and plan.attn_tower == key)
                streams[key] = s
        add_time, drop, mask = plan.embed
        pos = self.P["pos_emb"] if plan.learned_pos else self.sinus
        self.embed_fwd(ids, self.P["item_emb"], c.x0, pos=pos, add=streams["time"] if add_time else None,
                       rate=self.rate if (train and drop) else 0.0, site=SITE_EMBED, mask_ids=ids if mask else None)
        x = c.x0
        if plan.merge and plan.merge[3] == "pre":
            x = self.merge_fwd(c, {"seq": x, **streams}, ids, train)
        x = self.tower_fwd(c, "main", x, ids, train, want_attn and plan.attn_tower == "main")
        if plan.merge and plan.merge[3] == "post":
            x = self.merge_fwd(c, {"seq": x, **streams}, ids, train)
        c.seq_emb = x
        return x

    def loss_tail_fused(self, c):
        tb = c.tw["main"]
        H, N = self.H, c.N
        parts = self.lib.cast_lnf_loss_parts(N)
        self._call(self.lib.cast_lnf_loss, tb.x_last.data_ptr(), self.P["main.lnf.gamma"].data_ptr(),
                   self.P["main.lnf.beta"].data_ptr(), 1e-8, self.P["item_emb"].data_ptr(),
                   self.P["item_emb"].shape[0], H, N, c.keys3[1].data_ptr(), c.keys3[2].data_ptr(), tb.out.data_ptr(),
                   c.pos_logits.data_ptr(), c.neg_logits.data_ptr(), c.gpos.data_ptr(), c.gneg.data_ptr(),
                   c.t[0].data_ptr(), c.ws_tail.data_ptr(), c.ws_tail.numel() * 4, self._stream())
        base = c.ws_tail.data_ptr()
        c.reduce_jobs.append((base, parts, 3, c.sums, 3))
        c.reduce_jobs.append((base + 4 * 3 * parts, parts, H, self.G["main.lnf.gamma"], 2 * H))
        c.reduce_jobs.append((base + 4 * (3 * parts + H), parts, H, self.G["main.lnf.beta"], 2 * H))

    def loss_fwd_bwd(self, c, with_grad=True, defer_sums=False):
        ws, ws_bytes, sums = c.ws, c.ws_bytes, c.sums
        if defer_sums:  # the three loss sums join the step's single reduction launch (end of backward)
            ws, ws_bytes, sums = c.ws_loss, c.ws_loss.numel() * 4, None
            c.reduce_jobs.append((c.ws_loss.data_ptr(), self.lib.cast_logits_loss_parts(c.N), 3, c.sums, 3))
        tail = (c.keys3[1].data_ptr(), c.keys3[2].data_ptr(), c.pos_logits.data_ptr(), c.neg_logits.data_ptr(),
                self._p(sums), c.dseq.data_ptr() if with_grad else None, c.gpos.data_ptr() if with_grad else None,
                c.gneg.data_ptr() if with_grad else None, ws.data_ptr(), ws_bytes, self._stream())
        if self.item_shard is not None:
            self._call(self.lib.cast_logits_loss_sharded, c.seq_emb.data_ptr(), self.shard_ptrs.data_ptr(),
                       self.item_shard[1], self.V_items, self.H, c.N, *tail)
        else:
            self._call(self.lib.cast_logits_loss, c.seq_emb.data_ptr(), self.P["item_emb"].data_ptr(),
                       self.P["item_emb"].shape[0], self.H, c.N, *tail)

    def backward(self, c):
        """Un-normalised gradients of sum(loss terms) into self.g (the 1/sum(istarget) factor — global under data
        parallelism, models/sasrec.py:105-108 — is applied inside the Adam kernel)."""
        plan = self.plan
        ids = c.keys3[0]
        d = c.dseq
        dstreams: Dict[str, torch.Tensor] = {}
        if plan.merge and plan.merge[3] == "post":
            ds = self.merge_bwd(c, d)
            d = ds["seq"]
            dstreams.update({k: v for k, v in ds.items() if k != "seq"})
        add_time, drop, mask = plan.embed
        pre_merge = bool(plan.merge and plan.merge[3] == "pre")
        # the tower's input is dropout(emb) * mask: block 0's fused backward kernel applies that gradient itself
        fuse_embed = ((drop or mask) and not pre_merge and self.row_kernels
                      and len(c.tw["main"].blocks) > 0)
        d = self.tower_bwd(c, "main", d, ids, embed_fx=(ids if mask else None, self.rate if drop else 0.0, SITE_EMBED,
                                                        c.g0) if fuse_embed else None)
        if pre_merge:
            # cast_9's `seq *= mask` after the MLP (cast_9.py:174) needs no backward step: mlp_out is already masked,
            # so relu_bwd zeroes those rows (act == 0)
            ds = self.merge_bwd(c, d)
            d = ds["seq"]
            dstreams.update({k: v for k, v in ds.items() if k != "seq"})
        g0 = d
        if fuse_embed:
            g0 = c.g0
        elif drop or mask:
            self.mask_dropout(d, ids if mask else None, self.rate if drop else 0.0, SITE_EMBED, None, c.g0)
            g0 = c.g0
        if add_time:
            dstreams["time"] = g0
        if plan.learned_pos:
            th = self.T * self.H
            if self.row_kernels:
                # d(pos_emb) = sum over the batch of g0 [B, T*H]: another job of the step's reduction launch
                c.reduce_jobs.append((g0.data_ptr(), c.B, th, self.G["pos_emb"], th))
            else:
                self._call(self.lib.cast_colsum, g0.data_ptr(), c.B, th, th, self.G["pos_emb"].data_ptr(),
                           c.ws.data_ptr(), c.ws_bytes, self._stream())
        sq = float(self.H ** 0.5)
        ctx_scatter = []
        for j, (tname, key) in enumerate((("time_emb", "time"), ("hours_emb", "hours"), ("days_emb", "days"))):
            if tname not in plan.tables:
                continue
            dk = dstreams[key]
            if key in plan.towers:
                dk = self.tower_bwd(c, key, dk, ids)
            ctx_scatter.append((j, dk, tname))
        # every deferred partial sum of the step is known now: its one reduction launch runs beside the embedding
        # gradient scatters (independent outputs; a parallel branch of the captured graph), joined before the exchange
        if c.reduce_jobs:
            self._fork(c, "reduce", lambda: self.flush_reduce_jobs(c))
        self.scatter(c, c.keys3, 3, [g0, c.seq_emb, c.seq_emb], [None, c.gpos, c.gneg], [sq, 1.0, 1.0], "item_emb")
        for j, dk, tname in ctx_scatter:
            self.scatter(c, c.cids[j], 1, [dk], [None], [sq], tname)
        self._join(c, "reduce")
        self.flush_reduce_jobs(c)   # not forked: in stream order

    def rank_local(self):
        """context manager: steps launched inside touch no other rank (no barrier, exchange or peer reads) — for
        rank-local profiling; gradients are then this rank's own and the replicas drift apart, so callers restore state"""
        import contextlib

        @contextlib.contextmanager
        def cm():
            saved = (self.grad_allreduce, self.after_adam, self.before_backward, self.peer_adam, self.clip_peers)
            self.grad_allreduce = self.after_adam = self.before_backward = self.peer_adam = self.clip_peers = None
            try:
                yield self
            finally:
                self.grad_allreduce, self.after_adam, self.before_backward, self.peer_adam, self.clip_peers = saved
        return cm()

    def flush_reduce_jobs(self, c):
        """One fixed-order reduction launch for the per-CTA gradient partials of every fused backward kernel."""
        jobs = c.reduce_jobs
        if not jobs:
            return
        n = len(jobs)
        parts = (C.c_void_p * n)(*[int(j[0]) for j in jobs])
        nparts = (C.c_int * n)(*[int(j[1]) for j in jobs])
        counts = (C.c_long * n)(*[int(j[2]) for j in jobs])
        pitches = (C.c_long * n)(*[int(j[4]) for j in jobs])
        outs = (C.c_void_p * n)(*[j[3].data_ptr() for j in jobs])
        self._call(self.lib.cast_reduce_partials_batch, n, parts, nparts, counts, pitches, outs, self._stream())
        c.reduce_jobs = []

    def adam(self, c):
        # gradients are divided by sums[2] = sum(istarget) (global under data parallelism) inside the kernel; with a
        # row-sharded item table the flat buffers hold this rank's shard first, so the same launch updates it
        if self.clip:
            self.adam_clipped()
            return
        if self.stamp is not None:
            self.adam_lazy()
            return
        if self.peer_adam is not None:
            ptrs, n_ranks, g_red = self.peer_adam
            self._call(self.lib.cast_adam_tf_step_peers, self.w.data_ptr(), ptrs.data_ptr(), n_ranks, g_red.data_ptr(),
                       self.m.data_ptr(), self.v.data_ptr(), self.n_params, g_red.numel() - self.n_params, self.lr,
                       self.beta1, self.beta2, self.eps, self.l2, 0, self.l2_hi if self.l2 else 0,
                       self.adam_state.data_ptr(), self._stream())
            return
        self._call(self.lib.cast_adam_tf_step, self.w.data_ptr(), self.adam_g.data_ptr(), self.m.data_ptr(),
                   self.v.data_ptr(), self.n_params, self.lr, self.beta1, self.beta2, self.eps,
                   self.adam_g[self.n_params + 2:].data_ptr(), self.l2, 0, self.l2_hi if self.l2 else 0,
                   self.adam_state.data_ptr(), self._stream())

    def adam_lazy(self):
        """lazy_adam: the touched rows of the item table (or of this rank's shard), then dense TF-Adam over the rest of
        the flat buffer, which advances the beta powers once"""
        rows, region, n = self.P["item_emb"].shape[0], self.P["item_emb"].numel(), self.n_params
        if self.peer_adam is not None:
            ptrs, n_ranks, g_red = self.peer_adam
            sp, ep = self.peer_stamps
            self._call(self.lib.cast_adam_tf_rows_peers, self.w.data_ptr(), ptrs.data_ptr(), sp.data_ptr(),
                       ep.data_ptr(), n_ranks, self.m.data_ptr(), self.v.data_ptr(), rows, self.H, n, self.lr,
                       self.beta1, self.beta2, self.eps, self.adam_state.data_ptr(), self._stream())
            self._call(self.lib.cast_adam_tf_range_peers, self.w.data_ptr(), ptrs.data_ptr(), n_ranks, g_red.data_ptr(),
                       self.m.data_ptr(), self.v.data_ptr(), region, n, g_red.numel() - n, self.lr, self.beta1,
                       self.beta2, self.eps, self.adam_state.data_ptr(), self._stream())
            return
        g, gden = self.adam_g, self.adam_g[n + 2:].data_ptr()
        self._call(self.lib.cast_adam_tf_rows, self.w.data_ptr(), g.data_ptr(), self.m.data_ptr(), self.v.data_ptr(),
                   rows, self.H, self.lr, self.beta1, self.beta2, self.eps, gden, self.stamp.data_ptr(),
                   self.grad_epoch.data_ptr(), self.adam_state.data_ptr(), self._stream())
        self._call(self.lib.cast_adam_tf_range, self.w[region:].data_ptr(), g[region:].data_ptr(),
                   self.m[region:].data_ptr(), self.v[region:].data_ptr(), n - region, self.lr, self.beta1, self.beta2,
                   self.eps, gden, 0.0, 0, 0, self.adam_state.data_ptr(), 1, self._stream())

    def adam_clipped(self):
        """clip_grad: sum-of-squares passes over the gradient Adam consumes, one finalize launch that writes {scale,
        norm} to clip_out, then the update of adam() / adam_lazy() with g * scale.  Replicated data parallelism forms
        the rank-ordered sum into g_red in the sum-of-squares pass (the order of cast_adam_tf_step_peers) and updates
        from there; a row-sharded table's partials go to peer-visible memory, and one more barrier lets every rank fold
        all shards in rank order."""
        lib, P, n, H = self.lib, self.clip_nparts, self.n_params, self.H
        rows, region = self.P["item_emb"].shape[0], self.P["item_emb"].numel()
        lazy = self.stamp is not None
        l2_hi = self.l2_hi if self.l2 else 0       # lazy_adam refuses l2_emb, so 0 there
        w, m, v, st, clip = self.w, self.m, self.v, self.adam_state.data_ptr(), self.clip_out.data_ptr()
        part = lambda k: self.clip_parts.data_ptr() + 8 * P * k   # noqa: E731
        opt = (self.lr, self.beta1, self.beta2, self.eps)
        s = self._stream()
        if self.peer_adam is not None:
            ptrs, n_ranks, g_red = self.peer_adam
            lo = region if lazy else 0
            if lazy:
                sp, ep = self.peer_stamps
                self._call(lib.cast_clip_sumsq_rows_peers, ptrs.data_ptr(), sp.data_ptr(), ep.data_ptr(), n_ranks,
                           rows, H, n, part(1), s)
            self._call(lib.cast_clip_reduce_sumsq_peers, ptrs.data_ptr(), n_ranks, g_red.data_ptr(), w.data_ptr(), lo,
                       n, g_red.numel() - n, self.l2, 0, l2_hi, part(0), s)
            self._call(lib.cast_clip_finalize, part(0), (2 if lazy else 1) * P, None, 0, self.max_norm, clip, s)
            if lazy:
                self._call(lib.cast_adam_tf_rows_peers_clip, w.data_ptr(), ptrs.data_ptr(), sp.data_ptr(),
                           ep.data_ptr(), n_ranks, m.data_ptr(), v.data_ptr(), rows, H, n, *opt, clip, st, s)
            self._call(lib.cast_adam_tf_range_clip, w[lo:].data_ptr(), g_red[lo:].data_ptr(), m[lo:].data_ptr(),
                       v[lo:].data_ptr(), n - lo, *opt, g_red[n + 2:].data_ptr(), self.l2, 0, l2_hi, clip, st, 1, s)
            return
        g, gden = self.adam_g, self.adam_g[n + 2:].data_ptr()
        # the item table's partials: peer-visible with a row-sharded table that is attached, local otherwise
        peers = self.clip_peers if self.item_shard is not None else None
        tparts = self.clip_shard_parts.data_ptr() if peers is not None else part(1)
        if lazy:
            self._call(lib.cast_clip_sumsq_rows, g.data_ptr(), rows, H, gden, self.stamp.data_ptr(),
                       self.grad_epoch.data_ptr(), tparts, s)
        elif peers is not None:
            self._call(lib.cast_clip_sumsq_range, g.data_ptr(), w.data_ptr(), region, gden, self.l2, 0,
                       min(l2_hi, region), tparts, s)
        else:   # one pass over the whole buffer (part(1) stays zero)
            self._call(lib.cast_clip_sumsq_range, g.data_ptr(), w.data_ptr(), n, gden, self.l2, 0, l2_hi, part(0), s)
        if lazy or peers is not None:
            self._call(lib.cast_clip_sumsq_range, g[region:].data_ptr(), w[region:].data_ptr(), n - region, gden,
                       self.l2, 0, max(l2_hi - region, 0), part(0), s)
        if peers is not None:
            barrier, shard_ptrs = peers
            barrier()       # every rank's shard partials are final
            self._call(lib.cast_clip_finalize, part(0), P, shard_ptrs.data_ptr(), self.item_shard[1], self.max_norm,
                       clip, s)
        else:
            self._call(lib.cast_clip_finalize, part(0), (2 if lazy else 1) * P, None, 0, self.max_norm, clip, s)
        if lazy:
            self._call(lib.cast_adam_tf_rows_clip, w.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), rows, H,
                       *opt, gden, self.stamp.data_ptr(), self.grad_epoch.data_ptr(), clip, st, s)
            self._call(lib.cast_adam_tf_range_clip, w[region:].data_ptr(), g[region:].data_ptr(), m[region:].data_ptr(),
                       v[region:].data_ptr(), n - region, *opt, gden, 0.0, 0, 0, clip, st, 1, s)
        else:
            self._call(lib.cast_adam_tf_range_clip, w.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), n, *opt,
                       gden, self.l2, 0, l2_hi, clip, st, 1, s)

    def launch_fwd_bwd(self, c):
        # The sort of the (item id, entry) pairs for the embedding gradient depends on the ids only: it runs on a side
        # stream while the forward pass computes (a parallel branch of the captured CUDA graph) and is joined right
        # before the segment sums at the end of backward.
        def sort():
            if self.item_shard is not None:
                self._call(self.lib.cast_scatter_sort_sharded, c.keys3.data_ptr(), 3, c.N, self.V_items,
                           self.item_shard[1], self.shard_R, c.sws.data_ptr(), c.sws_bytes, self._stream())
            else:
                V = self.P["item_emb"].shape[0]
                self._call(self.lib.cast_scatter_sort, c.keys3.data_ptr(), 3, c.N, V, c.sws.data_ptr(), c.sws_bytes,
                           self._stream())

        try:
            if self._fork(c, "sort", sort) and self.rowk_img is not None:
                # the weight operand images are needed by the first row kernel, not by the embedding
                self._fork(c, "presplit", lambda: self.rowk_presplit(self._stream()))
            # "peers have finished reading the previous step's gradients": a flag round trip over NVLink that nothing in
            # the forward pass depends on => a parallel branch of the step, joined before the first gradient write
            if self.before_backward is not None:
                self._fork(c, "barrier", self.before_backward)
            self.forward(c, train=True)
            if self.before_backward is not None and not self._join(c, "barrier"):
                self.before_backward()
            if self.grad_epoch is not None:   # lazy_adam: the gradient rows this pass writes get a fresh stamp
                self._call(self.lib.cast_grad_epoch_advance, self.grad_epoch.data_ptr(), self._stream())
            if self.fuse_tail:
                self.loss_tail_fused(c)
            else:
                self.loss_fwd_bwd(c, with_grad=True, defer_sums=True)
            self.backward(c)
        finally:   # contexts are reused: a failed launch must leave no side branch un-joined and no deferred job behind
            for name in list(c.forked):
                self._join(c, name)
            c.reduce_jobs = []

    def launch_train_step(self, c):
        """Enqueue one full training step (forward, loss, backward, [gradient exchange], Adam) on the current stream."""
        self.launch_fwd_bwd(c)
        if self.grad_allreduce is not None:
            self.grad_allreduce(c)
        self.adam(c)
        if self.after_adam is not None:
            self.after_adam()
