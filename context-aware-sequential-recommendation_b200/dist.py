"""Data-parallel training over the GPUs of one box: one process per GPU.  `torch.distributed` only sets things up
(broadcast of the initial weights, exchange of the peer-memory handles, evaluation's final histogram sum); inside a
training step the ranks exchange gradients with plain kernel launches over NVLink peer mappings (PeerArena,
PeerExchange): a flag barrier, then every rank sums the ranks' buffers itself in rank order.  No collective call sits
in the step, so the whole step stays one CUDA graph.  With a row-sharded item table (BASELINE config 5) the table
traffic goes the same way: kernels read the owning rank's memory directly.

The reference is single-device (SURVEY §2.1); the semantics kept here are those of its loss: the gradient is the
derivative of  sum(loss terms) / sum(istarget)  over the WHOLE batch (models/sasrec.py:105-108).  Each rank therefore
contributes un-normalised gradient numerators plus its local sum(istarget); the rank-ordered sum over
[gradients | loss_sum, auc_sum, count] gives every rank the same global numerators and global denominator (the same
bits on every rank), and the Adam kernel divides.  N ranks with B/N sequences each reproduce the single-GPU step on
B sequences up to fp32 summation order.
"""
from __future__ import annotations

import os
from types import SimpleNamespace

import torch
import torch.distributed as dist


def init_from_env(backend: str | None = None):
    """torchrun / torch.distributed.run environment -> process group.  Returns (rank, world_size, local_rank)."""
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1 and not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29500")
        if backend is None:
            backend = "nccl" if torch.cuda.is_available() else "gloo"
        if backend == "nccl":
            torch.cuda.set_device(local)
        dist.init_process_group(backend=backend, rank=rank, world_size=world)
    return rank, world, local


class PeerArena:
    """Memory of this rank that the other ranks of the box read directly from their kernels (item-table shard, sorted
    gradient entries and their source rows): on GPUs ordinary device allocations whose CUDA IPC handles are exchanged
    through the process group and mapped with peer access (loads go over NVLink / NVSwitch, `cast_peer_open`); in the
    CPU tests (gloo, host-emulated kernels) POSIX shared memory.  `ptrs(t)` is a collective: every rank passes its own
    tensor and gets the address of each rank's tensor in ITS address space (own entry: the local pointer)."""

    def __init__(self, lib, device, group=None):
        self.lib, self.device, self.group = lib, torch.device(device), group
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        self._opened = {}      # IPC handle bytes / shm name -> base address in this process
        self._shm = []         # (SharedMemory, base address, size) segments this rank created
        self._keep = []

    def alloc(self, numel: int, dtype):
        """a zeroed buffer the other ranks can map: cudaMalloc + IPC handle (GPU) / named shared memory (CPU tests)"""
        import ctypes
        nbytes = max(256, int(numel) * torch.empty(0, dtype=dtype).element_size())
        if self.device.type == "cuda":
            ptr, handle = ctypes.c_void_p(), ctypes.create_string_buffer(64)
            rc = self.lib.cast_peer_alloc(nbytes, ctypes.byref(ptr), handle)
            if rc != 0:
                from . import _lib
                _lib.check(self.lib, rc, "cast_peer_alloc")
            base = int(ptr.value)

            class _Raw:   # torch wraps foreign device memory through the CUDA array interface (no copy, no ownership)
                __cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (base, False), "version": 2}

            t = torch.as_tensor(_Raw(), device=self.device)
            self._shm.append((("ipc", handle.raw), base, nbytes))
            return t.view(dtype)[:int(numel)]
        from multiprocessing import shared_memory
        shm = shared_memory.SharedMemory(create=True, size=nbytes)
        base = ctypes.addressof(ctypes.c_char.from_buffer(shm.buf))
        self._shm.append((shm, base, nbytes))
        return torch.frombuffer(shm.buf, dtype=dtype, count=int(numel))

    def _describe(self, t: torch.Tensor):
        p = t.data_ptr()
        for seg, base, nbytes in self._shm:
            if base <= p < base + nbytes:
                return (seg[0], seg[1], p - base) if isinstance(seg, tuple) else ("shm", seg.name, p - base)
        raise ValueError("PeerArena.ptrs: the tensor must come from PeerArena.alloc")

    def _open(self, kind, key):
        if key in self._opened:
            return self._opened[key]
        if kind == "ipc":
            import ctypes
            out = ctypes.c_void_p()
            rc = self.lib.cast_peer_open(key, ctypes.byref(out))
            if rc != 0:
                from . import _lib
                _lib.check(self.lib, rc, "cast_peer_open")
            base = int(out.value)
        else:
            from multiprocessing import shared_memory
            import ctypes
            shm = shared_memory.SharedMemory(name=key)
            self._keep.append(shm)
            base = ctypes.addressof(ctypes.c_char.from_buffer(shm.buf))
        self._opened[key] = base
        return base

    def ptrs(self, t: torch.Tensor):
        mine = self._describe(t)
        every = [None] * self.world
        dist.all_gather_object(every, mine, group=self.group)
        out = []
        for r, (kind, key, off) in enumerate(every):
            out.append(t.data_ptr() if r == self.rank else self._open(kind, key) + off)
        return out

    def close(self):
        for shm in self._keep:
            try:
                shm.close()
            except Exception:
                pass
        for seg, base, _ in self._shm:
            try:
                if isinstance(seg, tuple):
                    self.lib.cast_peer_free(base)
                else:
                    seg.close()
                    seg.unlink()
            except Exception:
                pass
        self._shm = []


class PeerExchange:
    """The step's cross-rank traffic as plain kernel launches over peer memory (no collective library inside the
    step, so the whole step is ONE CUDA graph): a flag barrier over NVLink (`cast_peer_barrier`) and the rank-ordered
    sum of the ranks' flat gradient buffers (`cast_peer_reduce`: every rank reads the n buffers and adds them in rank
    order => the same bits on every rank, reproducible run to run).  The engine's gradient buffer is re-homed into
    peer-visible memory; Adam and the loss read-back consume the reduced copy."""

    def __init__(self, engine, arena, group=None, first: int = 0):
        import ctypes as C
        self.eng, self.arena = engine, arena
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        self.first = int(first)               # elements before `first` are not reduced (a row-sharded table's gradient)
        dev = engine.device
        total = engine.gbuf.numel()
        gnew = arena.alloc(total, torch.float32)
        gnew.copy_(engine.gbuf)
        engine.rebind_gradients(gnew)
        self.count = total - self.first
        self.g_red = torch.zeros(total, dtype=torch.float32, device=dev)
        engine.adam_g = self.g_red
        gp = arena.ptrs(engine.gbuf)
        self.g_ptrs = torch.tensor([p + 4 * self.first for p in gp], dtype=torch.int64, device=dev)
        self.flags = arena.alloc(max(8, self.world), torch.int64)
        self.flag_ptrs = torch.tensor(arena.ptrs(self.flags), dtype=torch.int64, device=dev)
        self.state = torch.zeros(2, dtype=torch.int64, device=dev)

    def barrier(self):
        e = self.eng
        e._call(e.lib.cast_peer_barrier, self.flag_ptrs.data_ptr(), self.rank, self.world, self.state.data_ptr(),
                e._stream())

    def reduce(self):
        e = self.eng
        e._call(e.lib.cast_peer_reduce, self.g_ptrs.data_ptr(), self.world, self.count,
                self.g_red.data_ptr() + 4 * self.first, e._stream())

    def timed_out(self) -> bool:
        return bool(self.state[1].item())


def quiesce(engine, group=None):
    """No rank may release its peer memory (or exit) while another rank's last optimizer pass still reads it."""
    if engine.device.type == "cuda":
        torch.cuda.synchronize(engine.device)
    if dist.is_initialized():
        dist.barrier(group=group)


def _quiesce_at_exit(engine, group):
    import atexit

    def _at_exit():
        try:
            quiesce(engine, group)
        except Exception:
            pass

    atexit.register(_at_exit)


def attach(engine, group=None, arena=None):
    """Make `engine.launch_train_step` data parallel over `group` (default: the world group): replicated parameters;
    per step the ranks' [gradient numerators | loss_sum, auc_sum, count] buffers are summed in rank order.  A flag
    barrier over NVLink marks every rank's gradient buffer final; the Adam pass then reads the ranks' buffers over
    their peer mappings and adds them in rank order itself.  A second barrier, between the next step's forward and
    backward passes, keeps any rank from overwriting its buffer while a peer may still read it."""
    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        return engine
    if engine.item_shard is not None:
        return attach_sharded(engine, group, arena)
    engine.world_size = dist.get_world_size(group)
    engine.rank = dist.get_rank(group)
    # identical replicas: rank 0's parameters and optimizer state win
    for t in (engine.w, engine.m, engine.v, engine.adam_state):
        dist.broadcast(t, src=0, group=group)
    # independent dropout streams per rank (one global batch, different positions)
    engine.seed = (engine.seed + 0x9E3779B1 * engine.rank) & 0xFFFFFFFFFFFF

    arena = arena or PeerArena(engine.lib, engine.device, group)
    engine.arena = arena
    px = engine.peer_exchange = PeerExchange(engine, arena, group)

    # One barrier on the critical path: every rank's gradient buffer is final => Adam sums the ranks' buffers itself
    # (cast_adam_tf_step_peers).  The second barrier ("everybody has read everybody: the buffers may be overwritten")
    # is only needed before the NEXT backward pass writes gradients, so it sits between the next step's forward and
    # backward, where no rank waits for it.
    def exchange(c):
        px.barrier()

    engine.peer_adam = (px.g_ptrs, px.world, px.g_red)
    if engine.stamp is not None:
        # lazy_adam: every rank's Adam reads the ranks' row stamps and gradient epochs next to their gradient rows
        for name in ("stamp", "grad_epoch"):
            t = getattr(engine, name)
            shared = arena.alloc(t.numel(), t.dtype)
            shared.copy_(t)
            setattr(engine, name, shared)
        engine.peer_stamps = tuple(torch.tensor(arena.ptrs(t), dtype=torch.int64, device=engine.device)
                                   for t in (engine.stamp, engine.grad_epoch))
    engine.before_backward = px.barrier
    _quiesce_at_exit(engine, group)
    engine.grad_allreduce = exchange
    engine.exchange_capturable = True
    if engine.device.type == "cuda":
        torch.cuda.synchronize(engine.device)
    dist.barrier(group=group)
    return engine


def attach_sharded(engine, group=None, arena: "PeerArena | None" = None):
    """Data parallelism with the item table ROW-SHARDED over the ranks (BASELINE config 5; SURVEY §8e row 2).  Each rank
    holds 1/world of the table, of its gradient and of its Adam slots; the dense weights stay replicated.  Per step:

      forward / backward   the embedding, positive and negative lookups read rows from the owning rank's shard over
                           NVLink (peer mappings; no exchange step, no staging buffers); every rank sorts its
                           (item id, entry) pairs by (owner, local row) on a side stream
      exchange             a flag barrier (every rank's dense gradients, sorted entries and source rows are final),
                           then the rank-ordered sum of [dense-weight gradients | loss_sum, auc_sum, count] read
                           from the peers' buffers
      owner pull           each rank folds, rank by rank in rank order, the entries that hit ITS rows (read from the
                           peers' memory) into its dense gradient shard: fixed order, no atomics, no table collective
      TF-Adam              one launch over [own shard | dense weights]  (28 B/param of table traffic divided by world)
      barrier              shards are updated and the exported buffers may be overwritten

    The engine must have been built with item_shard=(rank, world)."""
    if engine.item_shard is None:
        raise ValueError("attach_sharded: build the engine with item_shard=(rank, world)")
    import ctypes as C
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    if engine.item_shard != (rank, world):
        raise ValueError(f"engine was built for shard {engine.item_shard}, process group says {(rank, world)}")
    engine.world_size, engine.rank = world, rank
    seeds = [None] * world
    dist.all_gather_object(seeds, int(engine.seed), group=group)
    if len(set(seeds)) != 1:   # each rank drew its rows of the table from the same stream only if the seeds agree
        raise ValueError(f"row-sharded item table: every rank must build the engine with the same seed, got {seeds}")
    arena = arena or getattr(engine, "arena", None)
    if arena is None:
        raise ValueError("attach_sharded: the engine's peer-visible buffers must come from a PeerArena "
                         "(Engine(..., item_shard=...) creates one when torch.distributed is initialised)")
    engine.arena = arena
    # dense weights and optimizer state: rank 0 wins; the table shards are consistent by construction (same draws)
    region = engine.P["item_emb"].numel()
    for t in (engine.w[region:], engine.m[region:], engine.v[region:], engine.adam_state):
        dist.broadcast(t, src=0, group=group)
    engine.seed = (engine.seed + 0x9E3779B1 * rank) & 0xFFFFFFFFFFFF
    shards = arena.ptrs(engine.w)          # the shard is the first tensor of the flat parameter buffer
    engine.shard_ptrs = torch.tensor(shards, dtype=torch.int64, device=engine.device)
    R, H = engine.shard_R, engine.H

    def build_peer_view(c):
        """pointers to every rank's sorted entries and source rows for this batch size (collective, first step only)"""
        nsrc, rows, rowscale, scale = c.shard_src
        ko, po = C.c_size_t(), C.c_size_t()
        engine.lib.cast_scatter_sorted_offsets(c.N, nsrc, world * R, C.byref(ko), C.byref(po))
        ws = arena.ptrs(c.sws)
        uniq = {}
        for t in rows + [r for r in rowscale if r is not None]:
            if id(t) not in uniq:
                uniq[id(t)] = arena.ptrs(t)
        view = []
        for p in range(world):
            rows_a = (C.c_void_p * nsrc)(*[uniq[id(t)][p] for t in rows])
            rs_a = (C.c_void_p * nsrc)(*[(uniq[id(t)][p] if t is not None else None) for t in rowscale])
            view.append((rows_a, rs_a, ws[p] + ko.value, ws[p] + po.value))
        stage = torch.empty(engine.lib.cast_scatter_stage_bytes(c.N, nsrc, H) // 4 + 16, dtype=torch.float32,
                            device=engine.device)
        # (the staged pass runs as ONE source of N*nsrc rows: its chunk partials need their own, larger scratch)
        spart = torch.empty(engine.lib.cast_scatter_partial_bytes(c.N * nsrc, 1, H) // 4 + 16, dtype=torch.float32,
                            device=engine.device)
        c.peer = SimpleNamespace(view=view, scale=(C.c_float * nsrc)(*scale), nsrc=nsrc, stage=stage, spart=spart)

    px = engine.peer_exchange = PeerExchange(engine, arena, group, first=region)
    engine.exchange_capturable = True

    def exchange(c):
        px.barrier()    # every rank's dense gradients, sorted entries and source rows are final
        px.reduce()     # dense gradients + loss sums, rank order
        if c.peer is None:
            build_peer_view(c)
        pv = c.peer
        # lazy_adam: the owner's stamps decide write or add per row (no zeroing pass, no accumulate flag)
        lazy = (engine.stamp.data_ptr(), engine.grad_epoch.data_ptr()) if engine.stamp is not None else None
        for p in range(world):
            rows_a, rs_a, keys_p, pay_p = pv.view[p]
            if lazy and p == rank:
                engine._call(engine.lib.cast_scatter_apply_range_lazy, pv.nsrc, c.N, rows_a, rs_a, pv.scale, H,
                             engine.adam_g.data_ptr(), keys_p, pay_p, rank * R, (rank + 1) * R, c.spart.data_ptr(),
                             c.spart_bytes, *lazy, engine._stream())
            elif lazy:
                engine._call(engine.lib.cast_scatter_pull_range_lazy, pv.nsrc, c.N, rows_a, rs_a, pv.scale, H,
                             engine.adam_g.data_ptr(), keys_p, pay_p, rank * R, (rank + 1) * R, pv.stage.data_ptr(),
                             pv.stage.numel() * 4, pv.spart.data_ptr(), pv.spart.numel() * 4, *lazy, engine._stream())
            elif p == rank:   # own entries: summed straight from the source rows
                engine._call(engine.lib.cast_scatter_apply_range, pv.nsrc, c.N, rows_a, rs_a, pv.scale, H,
                             engine.adam_g.data_ptr(), keys_p, pay_p, rank * R, (rank + 1) * R, c.spart.data_ptr(),
                             c.spart_bytes, 1 if p else 0, engine._stream())
            else:           # a peer's entries: gathered over NVLink with one warp per row, then summed locally
                engine._call(engine.lib.cast_scatter_pull_range, pv.nsrc, c.N, rows_a, rs_a, pv.scale, H,
                             engine.adam_g.data_ptr(), keys_p, pay_p, rank * R, (rank + 1) * R, pv.stage.data_ptr(),
                             pv.stage.numel() * 4, pv.spart.data_ptr(), pv.spart.numel() * 4, 1 if p else 0,
                             engine._stream())

    engine.grad_allreduce = exchange
    engine.after_adam = px.barrier   # shards are updated; exported buffers may be overwritten
    if engine.clip:
        # clip_grad: every rank folds every rank's shard partials (peer mappings) after one more barrier
        engine.clip_peers = (px.barrier, torch.tensor(arena.ptrs(engine.clip_shard_parts), dtype=torch.int64,
                                                      device=engine.device))
    if engine.device.type == "cuda":
        torch.cuda.synchronize(engine.device)
    dist.barrier(group=group)      # every shard is initialised before anybody gathers from it
    return engine


def shard_users(n_users: int, rank: int, world: int):
    """Contiguous user shard for evaluation (users are independent; SURVEY §8e)."""
    per = (n_users + world - 1) // world
    lo = min(n_users, rank * per)
    return lo, min(n_users, lo + per)


def reduce_rank_histogram(hist: torch.Tensor, group=None):
    """Evaluation's only exchange: int64 histogram of ranks 0..9 + valid-user count (integers => exact HR@10)."""
    if dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(hist, op=dist.ReduceOp.SUM, group=group)
    return hist
