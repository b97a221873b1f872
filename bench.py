#!/usr/bin/env python
"""bench.py — train sequences/s of the SASRec hot path on ml-1m-shaped synthetic data (BASELINE.json configs[1]:
6040 users, 3416 items, maxlen 200, hidden 50, 2 blocks, 1 head, dropout 0.2; per-GPU batch 128 = the reference's
ml-1m run, saved_models/ml-1m.txt/sasrec_baseline_*/params.txt), full training step = forward + loss + backward +
deterministic sparse embedding gradient + (all-reduce) + TF-Adam.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--batch_size B] [--impl reference] [--dump-outputs DIR]

Prints ONE JSON line (rank 0).  `value` = whole-job sequences/s with inputs resident in HBM (CUDA-graph replay, CUDA
events, max over ranks, L2 flushed between timed steps); `e2e` = the same through `SASRec.train_step(sync=False)` with HOST
numpy batches (pinned staging + H2D + D2H of the loss inside the timed region); `roofline` = the dominant kernel
timed with CUDA events on the launch stream; `cpu_baseline` = the CPU oracle (PyTorch restatement of the reference
graph, `oracle/`) on the box's host cores over a bounded sample.  `--impl reference` times that CPU arm alone.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from types import SimpleNamespace

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# BASELINE.json configs (SURVEY §8): the metric is quoted on C2; the others are selectable with --config
CONFIGS = {
    "c2": dict(model="sasrec", users=6040, items=3416, mean_len=163.5, T=200, H=50, L=2, h=1, drop=0.2,
               desc="C2: SASRec ml-1m-shaped synthetic (6040 users, 3416 items, mean train len 163.5), maxlen=200, "
                    "hidden=50, blocks=2, heads=1, dropout=0.2"),
    "c1": dict(model="sasrec", users=52024, items=57289, mean_len=7.6, T=50, H=50, L=2, h=1, drop=0.5,
               desc="C1: SASRec Beauty-shaped synthetic (52024 users, 57289 items, mean len 7.6), maxlen=50, hidden=50, "
                    "blocks=2, heads=1, dropout=0.5"),
    "c3": dict(model="cast_1", users=6040, items=3416, mean_len=163.5, T=200, H=50, L=2, h=2, drop=0.2,
               desc="C3: CAST (cast_1, time-context tower) on ml-1m-shaped synthetic data with time bins, maxlen=200, "
                    "hidden=50, blocks=2, heads=2, dropout=0.2"),
    "c4": dict(model="sasrec", users=300000, items=30000, mean_len=12.0, T=50, H=128, L=4, h=4, drop=0.2,
               desc="C4: Steam/Video-shaped synthetic (300k users, 30k items, mean len 12), maxlen=50, hidden=128, "
                    "blocks=4, heads=4, dropout=0.2"),
    "c5": dict(model="sasrec", users=10000000, items=1000000, mean_len=100.0, T=200, H=256, L=2, h=1, drop=0.2,
               desc="C5: synthetic large catalog (10M users, 1M items, mean len 100), maxlen=200, hidden=256, blocks=2, "
                    "heads=1, dropout=0.2"),
}
CFG = CONFIGS["c2"]
WORKLOAD, USERNUM, ITEMNUM, MEAN_LEN = CFG["desc"], CFG["users"], CFG["items"], CFG["mean_len"]


def select_config(name):
    global CFG, WORKLOAD, USERNUM, ITEMNUM, MEAN_LEN
    CFG = CONFIGS[name]
    WORKLOAD, USERNUM, ITEMNUM, MEAN_LEN = CFG["desc"], CFG["users"], CFG["items"], CFG["mean_len"]


def make_args(batch_size):
    return SimpleNamespace(hidden_units=CFG["H"], maxlen=CFG["T"], num_heads=CFG["h"], num_blocks=CFG["L"],
                           num_context_blocks=2, max_bins=200, l2_emb=0.0, lr=1e-3, dropout_rate=CFG["drop"], seed=42,
                           batch_size=batch_size, bin_in_hours=48, log_scale=False)


def synth_batches(n_batches, B, T, itemnum, seed):
    """Seeded ml-1m-shaped batches in the sampler's layout (left-padded seq/pos/neg; sampler.py:16-81): lognormal
    lengths matched to the 163.5 mean train length (test.py:32-34), Zipf(1.0) item popularity."""
    rng = np.random.RandomState(seed)
    ranks = np.arange(1, itemnum + 1, dtype=np.float64)
    prob = ranks ** -1.0
    prob /= prob.sum()
    cdf = np.cumsum(prob)
    cdf[-1] = 1.0
    out = []
    for _ in range(n_batches):
        seq = np.zeros((B, T), np.int32)
        pos = np.zeros((B, T), np.int32)
        neg = np.zeros((B, T), np.int32)
        lens = np.clip(rng.lognormal(np.log(MEAN_LEN) - 0.32, 0.8, B), 3, 2000).astype(np.int64)
        for b in range(B):
            n = int(min(lens[b], T + 1))
            items = np.searchsorted(cdf, rng.rand(n)) + 1
            k = n - 1
            seq[b, T - k:] = items[:-1][-k:] if k else []
            pos[b, T - k:] = items[1:][-k:] if k else []
            neg[b, T - k:] = rng.randint(1, itemnum + 1, k)
        live = seq > 0
        ts = np.where(live, np.minimum(200, rng.geometric(0.05, (B, T)) - 1), 0).astype(np.int32)
        ts[:, -1] = 0  # the newest event is always in bin 0 (sampler.py:61-72)
        hrs = np.where(live, rng.randint(1, 25, (B, T)), 0).astype(np.int32)
        dys = np.where(live, rng.randint(1, 8, (B, T)), 0).astype(np.int32)
        out.append((seq, pos, neg, ts, hrs, dys))
    return out


class ClockSampler:
    """SM clock / throttle reasons while the timed region runs (B200_PROFILING.md recipe).  NVML is polled in-process
    every few ms (a 50-step region lasts ~30 ms: an `nvidia-smi -lms` child often reports nothing before it is over);
    `nvidia-smi` is the fallback when the NVML binding is missing."""

    REASONS = ((0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"), (0x4, "sw_power_cap"))

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.gpu = [], None, gpu_index
        self.nvml = self.handle = self.thread = None
        self.stop_flag = threading.Event()
        self.max_mhz = None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = gpu_index
            if vis:   # NVML enumerates every GPU of the box, CUDA only the visible ones
                ent = [v.strip() for v in vis.split(",") if v.strip()]
                if gpu_index < len(ent) and ent[gpu_index].isdigit():
                    idx = int(ent[gpu_index])
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def sample_now(self):
        """one NVML reading from the calling thread (the timed loop calls it half-way: at least one sample is inside the
        region however short it is)"""
        nv = self.nvml
        if nv is None:
            return
        try:
            mhz = float(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM))
            try:
                mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
            except Exception:
                mask = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
            self.rows.append((mhz, mask))
        except Exception:
            pass

    def _poll(self):
        while not self.stop_flag.is_set():
            self.sample_now()
            time.sleep(0.002)

    def start(self):
        if self.nvml is not None:
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.nvml is not None:
            self.stop_flag.set()
            self.thread.join(timeout=1)
            sm = [r[0] for r in self.rows]
            reasons = sorted({name for _, m in self.rows for bit, name in self.REASONS if m & bit})
            return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.max_mhz, "reasons": reasons,
                    "samples": len(sm), "source": "nvml"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"),
                                   r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "source": "nvidia-smi"}


def cpu_reference_arm(batch_size, steps, warmup, seed=20191019):
    """The reference's CPU path for this workload = oracle (PyTorch-CPU restatement; TF 1.15 is not installable):
    forward + backward + TF-Adam on all host cores."""
    from oracle import cast_oracle as O
    args = make_args(batch_size)
    torch.set_num_threads(os.cpu_count() or 1)
    p = O.init_params(CFG["model"], args, ITEMNUM, seed=42)
    opt = O.TFAdam(p, lr=args.lr)
    batches = synth_batches(2, batch_size, args.maxlen, ITEMNUM, seed)
    gen = torch.Generator().manual_seed(1)

    def drop(site, x):
        keep = (torch.rand(x.shape, generator=gen) >= args.dropout_rate).to(x.dtype)
        return x * keep / (1.0 - args.dropout_rate)

    def step(i):
        seq, pos, neg, ts, hrs, dys = batches[i % len(batches)]
        b = {"input_seq": torch.from_numpy(seq), "pos": torch.from_numpy(pos), "neg": torch.from_numpy(neg),
             "time_seq": torch.from_numpy(ts), "hours": torch.from_numpy(hrs), "days": torch.from_numpy(dys)}
        return O.train_step(CFG["model"], p, opt, args, b, drop)

    for i in range(warmup):
        step(i)
    t0 = time.perf_counter()
    for i in range(steps):
        step(i)
    dt = time.perf_counter() - t0
    return batch_size * steps / dt, dt / steps, torch.get_num_threads()


DP_PARITY_TOL = 2e-5


def dp_parity_check(model, eng, c, dev_batches, B, world, rank, dev, shard):
    """(1) every rank holds bit-identical replicated parameters after the timed steps; (2) gradients of ONE data-parallel
    step over N x B sequences equal (2e-5 of each tensor's max) those of the same N x B sequences processed by a single
    rank without any exchange — dense weights through the all-reduce, item-table rows through whichever path the run
    uses (replicated scatter or, row-sharded, the owner pull over peer memory).  Dropout is off for (2): ranks draw
    independent masks by design."""
    import torch.distributed as dist
    region = eng.P["item_emb"].numel() if shard else 0
    wi = eng.w[region:].view(torch.int32).long()
    chk = torch.stack([wi.sum(), (wi * (torch.arange(wi.numel(), device=dev) % 8191 + 1)).sum()])
    allchk = [torch.zeros_like(chk) for _ in range(world)]
    dist.all_gather(allchk, chk)
    identical = all(bool(torch.equal(allchk[0], x)) for x in allchk)
    saved = (eng.w.clone(), eng.m.clone(), eng.v.clone(), eng.adam_state.clone(), eng.rate)
    eng.rate = 0.0
    k3, c3 = dev_batches[0]
    c.keys3.copy_(k3)
    c.cids.copy_(c3)
    eng.launch_fwd_bwd(c)
    eng.grad_allreduce(c)
    if eng.peer_adam is not None:    # the rank-ordered sum happens inside the optimizer pass, which leaves it in adam_g
        eng.adam(c)
    torch.cuda.synchronize(dev)
    g_dp = eng.adam_g.clone()        # the exchanged gradients (what Adam consumes)
    if eng.peer_adam is not None:
        eng.w.copy_(saved[0]); eng.m.copy_(saved[1]); eng.v.copy_(saved[2]); eng.adam_state.copy_(saved[3])
    # the same global batch on every rank, no exchange
    gk3 = [torch.zeros_like(k3) for _ in range(world)]
    gc3 = [torch.zeros_like(c3) for _ in range(world)]
    dist.all_gather(gk3, k3)
    dist.all_gather(gc3, c3)
    cg = eng.ctx(B * world)
    cg.keys3.copy_(torch.cat([x.view(3, B, -1) for x in gk3], 1).reshape(3, -1))
    cg.cids.copy_(torch.cat([x.view(3, B, -1) for x in gc3], 1).reshape(3, -1))
    eng.launch_fwd_bwd(cg)
    if shard:   # own rows of the gradient from this rank's own sorted entries (they cover the whole batch now)
        import ctypes as C
        nsrc, rows, rowscale, scale = cg.shard_src
        ko, po = C.c_size_t(), C.c_size_t()
        eng.lib.cast_scatter_sorted_offsets(cg.N, nsrc, world * eng.shard_R, C.byref(ko), C.byref(po))
        rows_a = (C.c_void_p * nsrc)(*[t.data_ptr() for t in rows])
        rs_a = (C.c_void_p * nsrc)(*[(t.data_ptr() if t is not None else None) for t in rowscale])
        eng._call(eng.lib.cast_scatter_apply_range, nsrc, cg.N, rows_a, rs_a, (C.c_float * nsrc)(*scale), eng.H,
                  eng.G["item_emb"].data_ptr(), cg.sws.data_ptr() + ko.value, cg.sws.data_ptr() + po.value,
                  rank * eng.shard_R, (rank + 1) * eng.shard_R, cg.spart.data_ptr(), cg.spart_bytes, 0, eng._stream())
    torch.cuda.synchronize(dev)
    g_1 = eng.gbuf.clone()
    worst, worst_name = 0.0, ""
    for name, off in eng.offsets.items():
        if name.endswith("k.b"):      # analytically zero (softmax shift invariance): rounding noise only
            continue
        n = eng.P[name].numel()
        a_, b_ = g_dp[off:off + n], g_1[off:off + n]
        e = float((a_ - b_).abs().max() / b_.abs().max().clamp_min(1e-30))
        if e > worst:
            worst, worst_name = e, name
    sums_ok = bool(g_dp[-2] == g_1[-2]) and abs(float(g_dp[-4] - g_1[-4])) <= DP_PARITY_TOL * abs(float(g_1[-4]))
    t = torch.tensor([worst, 0.0 if sums_ok else 1.0, 0.0 if identical else 1.0], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    eng.w.copy_(saved[0]); eng.m.copy_(saved[1]); eng.v.copy_(saved[2]); eng.adam_state.copy_(saved[3])
    eng.rate = saved[4]
    if eng.after_adam is not None:
        eng.after_adam()
    worst = float(t[0].item())
    # fp32 association only: the N ranks' partial sums are added in rank order, the single rank sums the N x B rows in
    # its own order; measured 1.1e-6 / 2.5e-6 / 5.6e-6 at N = 2 / 4 / 8 (a broken exchange shows up as O(1))
    ok = worst <= DP_PARITY_TOL and t[1].item() == 0 and t[2].item() == 0
    return {"ok": bool(ok), "replicas_bit_identical": bool(t[2].item() == 0), "grad_max_rel_err_vs_single_rank": worst,
            "worst_tensor_rank0": worst_name, "loss_and_count_match": bool(t[1].item() == 0), "tolerance": DP_PARITY_TOL,
            "global_batch": B * world, "item_table": "row-sharded" if shard else "replicated"}


DUMP_LIMIT_BYTES = 64 << 20
DUMP_TABLE_ROWS = 16384


def dump_outputs(out_dir, eng):
    """Writes what the last timed step handed its caller, as DIR/<name>.npy: `loss` and `auc` (float64, the values
    `train_step` returns) and `param.<role name>` (float32, every parameter after the step's optimizer update).  A
    table with more than DUMP_TABLE_ROWS rows is cut to a fixed seeded sample of its rows, the same rows on every run,
    so that the outputs of two builds can be compared file by file."""
    loss_sum, auc_sum, cnt = eng.global_sums()[:3].tolist()
    arrays = {"loss": np.float64(loss_sum / cnt), "auc": np.float64(auc_sum / cnt)}
    for name, t in eng.P.items():
        if t.dim() == 2 and t.shape[0] > DUMP_TABLE_ROWS:   # rows picked on the device: only the sample is copied
            rows = np.sort(np.random.RandomState(0).choice(t.shape[0], DUMP_TABLE_ROWS, replace=False))
            t = t[torch.from_numpy(rows).to(t.device)]
        arrays["param." + name] = t.cpu().numpy()
    total = sum(v.nbytes for v in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError(f"--dump-outputs would write {total} bytes (limit {DUMP_LIMIT_BYTES})")
    os.makedirs(out_dir, exist_ok=True)
    for name, v in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), v)


def bench_config(batch_per_gpu, gpus):
    """the workload both arms name (identical dict in both lines; how each arm ran it is under `notes` / `sample`)"""
    return {"workload": WORKLOAD, "batch_per_gpu": batch_per_gpu, "global_batch": batch_per_gpu * gpus}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch_size", type=int, default=128, help="per-GPU batch (weak scaling)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS), help="BASELINE.json workload (default: the "
                    "one the metric is quoted on)")
    ap.add_argument("--model", default=None, help="override the config's model (e.g. --config c3 --model cast_4)")
    ap.add_argument("--cpu_steps", type=int, default=8)
    ap.add_argument("--no_cpu_baseline", action="store_true")
    ap.add_argument("--no_profile", action="store_true")
    ap.add_argument("--no_eval", action="store_true")
    ap.add_argument("--shard_item_table", action="store_true", help="row-shard the item table across ranks: 1/N of the "
                    "table, its gradient and Adam slots per GPU, lookups over NVLink peer memory (default for "
                    "--config c5 when --gpus > 1)")
    ap.add_argument("--no_dp_parity", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the loss, AUC and parameters "
                    "of the last timed step (rank 0) as DIR/<name>.npy; same arguments, same inputs")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    select_config(a.config)
    if a.model:
        global WORKLOAD
        CFG["model"] = a.model
        CFG["desc"] = CFG["desc"] + f" [model {a.model}]"
        WORKLOAD = CFG["desc"]
    a.warmup = max(a.warmup, 3)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if a.impl == "reference":
        if rank != 0:
            return
        v, sps, cores = cpu_reference_arm(a.batch_size, a.steps, a.warmup)
        sample = (f"{a.steps} timed training steps (after {a.warmup} warm-up steps) of B={a.batch_size} sequences "
                  f"(fwd+bwd+TF-Adam) on the box's host cores, PyTorch-CPU oracle; one process whatever --gpus says")
        print(json.dumps({
            "impl": "reference", "metric": "train_seqs_per_sec", "value": v, "unit": "seq/s", "n_gpus": a.gpus,
            "steps": a.steps, "warmup": a.warmup, "ms_per_step": sps * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": bench_config(a.batch_size, a.gpus),
            "cpu_baseline": {"value": v, "unit": "seq/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": "seq/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    import cast_b200
    from cast_b200 import dist as cdist
    rank, world, local = cdist.init_from_env()
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    args = make_args(a.batch_size)
    B, T, H = a.batch_size, args.maxlen, args.hidden_units
    shard = world > 1 and (a.shard_item_table or a.config == "c5")
    model = cast_b200.build_model(CFG["model"], USERNUM, ITEMNUM, 5, args, device=dev, use_graph=True,
                                  item_shard=(rank, world) if shard else None)
    eng = model.engine
    cdist.attach(eng)
    lib = eng.lib
    batches = synth_batches(8, B, T, ITEMNUM, seed=20191019 + 1000 * rank)
    c = eng.ctx(B)

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize(dev)

    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)  # > 126 MB L2

    # ---- (1) device-resident throughput: inputs already in HBM, graph replay, per-step CUDA events
    dev_batches = [(torch.from_numpy(np.stack([x.reshape(-1) for x in b[:3]])).to(dev),
                    torch.from_numpy(np.stack([x.reshape(-1) for x in b[3:]])).to(dev)) for b in batches]
    model.train_step(None, *batches[0])  # builds buffers, captures the graph(s)
    n0 = lib.cast_launch_count()
    model.train_step(None, *batches[1])
    launches_eager = lib.cast_launch_count() - n0  # 0 under graph replay
    launches_per_step = getattr(model, "launches_per_step", None) or launches_eager

    def device_step(i):
        k3, c3 = dev_batches[i % len(dev_batches)]
        c.keys3.copy_(k3)
        c.cids.copy_(c3)
        model.launch(c)

    for i in range(a.warmup):
        device_step(i)
    barrier()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(a.steps)]
    barrier()
    for i in range(a.steps):
        flush.zero_()
        ev[i][0].record()
        device_step(i)
        ev[i][1].record()
        if rank == 0 and i == a.steps // 2:
            clocks.sample_now()
    barrier()
    clk = clocks.stop() if rank == 0 else None
    t_dev = sum(s.elapsed_time(e) for s, e in ev) / 1e3
    t = torch.tensor([t_dev], dtype=torch.float64, device=dev)
    t_dev_min = t_dev
    if world > 1:
        tmin = t.clone()
        torch.distributed.all_reduce(tmin, op=torch.distributed.ReduceOp.MIN)
        t_dev_min = float(tmin.item())
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    t_dev = float(t.item())
    value = world * B * a.steps / t_dev
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, eng)

    # ---- (2) end to end through the public API with host batches
    for i in range(3):
        model.train_step(None, *batches[i % len(batches)])
    barrier()
    t0 = time.perf_counter()
    for i in range(a.steps):   # every step: pinned staging + H2D of its batch, the step, D2H of its {loss, auc, count};
        model.train_step(None, *batches[i % len(batches)], sync=False)   # the host reads step i-1's while step i runs
    e2e_last = model.last_metrics()
    torch.cuda.synchronize(dev)
    t_e2e = time.perf_counter() - t0
    assert e2e_last is not None and np.isfinite(e2e_last[1])
    t = torch.tensor([t_e2e], dtype=torch.float64, device=dev)
    if world > 1:
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    t_e2e = float(t.item())
    e2e = {"value": world * B * a.steps / t_e2e, "unit": "seq/s", "h2d_bytes_per_step": (6 if len(eng.plan.tables) > 1 else 3) * B * T * 4,
           "d2h_bytes_per_step": 12, "ms_per_step": t_e2e / a.steps * 1e3}

    # ---- (2b) evaluation throughput (BASELINE metric "eval users/sec"): host candidate arrays in, ranks out, through
    # the public batched API — forward at maxlen 200 + 101-candidate scoring, and the full-catalog tcgen05 ranking
    eval_out = None
    if not a.no_eval and CFG["model"].startswith("sasrec"):
        # users are sharded over the ranks (each rank scores its own users; SURVEY §8e); with a row-sharded item table
        # the full-catalog mode is a collective: all-gathered user vectors x own item shard + one integer all-reduce
        rs = np.random.RandomState(7 + rank)
        EU, EB = 2048, 512       # users per rank, users per call
        if CFG["items"] > 200000:
            EU, EB = 512, 256
        eseq = np.concatenate([b[0] for b in synth_batches(max(1, EU // B), B, T, ITEMNUM, seed=99 + rank)], 0)[:EU]
        EU = eseq.shape[0]
        ecand = rs.randint(1, ITEMNUM + 1, (EU, 101)).astype(np.int32)
        res = {}
        for name, fn in (("101", lambda s_, c_: model.score_candidates(s_, c_)),
                         ("full", lambda s_, c_: model.score_full_catalog(s_, c_[:, 0]))):
            fn(eseq[:EB], ecand[:EB])  # warm (buffers, smem attributes)
            barrier()
            t0 = time.perf_counter()
            for s0 in range(0, EU, EB):
                fn(eseq[s0:s0 + EB], ecand[s0:s0 + EB])
            torch.cuda.synchronize(dev)
            tt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
            if world > 1:
                torch.distributed.all_reduce(tt, op=torch.distributed.ReduceOp.MAX)
            res[name] = world * EU / float(tt.item())
        eval_out = {"users_per_sec_101": res["101"], "users_per_sec_full_catalog": res["full"], "users": EU * world,
                    "batch_users": EB, "unit": "users/s", "ranks": world, "catalog_items": ITEMNUM,
                    "item_table": "row-sharded" if shard else "replicated",
                    "note": "users sharded over the ranks, whole-job users / max-over-ranks wall time; host int32 "
                            "arrays in, ranks out (H2D + forward + scoring + D2H inside the timed region)"}

    # ---- (2a') where a multi-GPU step goes: [forward+backward graph | exchange | Adam graph | end-of-step barrier]
    step_split = None
    if world > 1:
        # eager launches of the same kernels, one CUDA event per segment (in the timed runs the step is one graph)
        names = ("fwd_bwd", "exchange", "adam", "end_of_step_barrier")
        acc = torch.zeros(4, dtype=torch.float64, device=dev)
        nrep = 5
        for i in range(nrep + 2):
            k3, c3 = dev_batches[i % len(dev_batches)]
            c.keys3.copy_(k3)
            c.cids.copy_(c3)
            evs = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
            evs[0].record()
            eng.launch_fwd_bwd(c)
            evs[1].record()
            if eng.grad_allreduce is not None:
                eng.grad_allreduce(c)
            evs[2].record()
            eng.adam(c)
            evs[3].record()
            if eng.after_adam is not None:
                eng.after_adam()
            evs[4].record()
            torch.cuda.synchronize(dev)
            if i >= 2:
                acc += torch.tensor([evs[j].elapsed_time(evs[j + 1]) for j in range(4)], dtype=torch.float64, device=dev)
        acc /= nrep
        mx = acc.clone()
        torch.distributed.all_reduce(mx, op=torch.distributed.ReduceOp.MAX)
        mn = acc.clone()
        torch.distributed.all_reduce(mn, op=torch.distributed.ReduceOp.MIN)
        step_split = {n: {"max_ms": float(a_), "min_ms": float(b_)} for n, a_, b_ in zip(names, mx.tolist(), mn.tolist())}
        step_split["note"] = ("eager launches (the timed step replays them as one CUDA graph), L2 not flushed; a rank "
                              "that finishes its backward pass early waits inside `exchange` for the slowest one: "
                              "min over ranks is the exchange itself")
        step_split["exchange_is"] = (("flag barrier + rank-ordered sum of the dense gradients over peer memory" if
                                      eng.exchange_capturable else "process-group all-reduce of the dense gradients") +
                                     (" + owner pull of the item-table rows over NVLink (one staged gather + local "
                                      "segment sums per peer, rank order)" if shard else ""))

    # ---- (2c) data-parallel parity ON THE BOX (world > 1): replicas bit-identical after the timed steps, and one
    # N-rank step == the same global batch processed by one rank (dropout off: ranks draw independent masks)
    dp_parity = None
    if world > 1 and not a.no_dp_parity:
        dp_parity = dp_parity_check(model, eng, c, dev_batches, B, world, rank, dev, shard)

    # ---- (3) per-kernel CUDA-event profile (eager launches on the same stream) -> dominant kernel roofline
    roofline, kernels = None, None
    if rank == 0 and not a.no_profile:
        from cast_b200 import profile as cprof
        kernels = cprof.profile_step(model, c, steps=min(a.steps, 10))
        roofline = cprof.roofline_of_dominant(kernels, B, T, H, args, ROOT)

    out = {"metric": "train_seqs_per_sec", "value": value, "unit": "seq/s", "n_gpus": world, "steps": a.steps,
           "warmup": a.warmup, "ms_per_step": t_dev / a.steps * 1e3, "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": bench_config(B, world),
           "notes": {"parallelism": f"dp{world}" + ("+item-table-row-sharded(1/%d per GPU, NVLink peer gathers, "
                                                     "owner-pull gradient)" % world if shard else ""),
                     "l2": "flushed (256 MiB write) between timed steps",
                     "timing": "per-step CUDA events on the launch stream, max over ranks",
                     "ms_per_step_fastest_rank": t_dev_min / a.steps * 1e3,
                     "input_path": "pre-generated synthetic batches (not the reference sampler)"},
           "e2e": e2e, "gpu_launches": int(launches_per_step) * a.steps, "launches_per_step": int(launches_per_step),
           "clocks": clk}
    if eval_out is not None:
        out["eval"] = eval_out
    if dp_parity is not None:
        out["dp_parity"] = dp_parity
    if step_split is not None:
        out["step_split"] = step_split
    out["hbm_per_gpu"] = {"params_mb": eng.w.numel() * 4 / 1e6, "item_table_rows_local": int(eng.P["item_emb"].shape[0]),
                          "item_table_rows_total": ITEMNUM + 1}
    if roofline is not None:
        out["roofline"] = roofline
        out["kernel_profile"] = kernels
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        v, sps, cores = cpu_reference_arm(B, a.cpu_steps, 1)
        out["cpu_baseline"] = {"value": v, "unit": "seq/s", "cores": cores, "kind": "port",
                               "sample": f"{a.cpu_steps} training steps of B={B} (fwd+bwd+TF-Adam), PyTorch-CPU oracle"}
    if rank == 0:
        print(json.dumps(out), flush=True)
    if world > 1:
        cdist.quiesce(eng)
        torch.distributed.destroy_process_group()
    if dp_parity is not None and not dp_parity["ok"]:
        sys.exit(3)


if __name__ == "__main__":
    main()
