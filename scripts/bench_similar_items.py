#!/usr/bin/env python
"""Benchmark of the all-items similar-items job (cast_similar_items: every item's top K neighbours, itself excluded) on a
seeded random item table, both metrics, with cast_topk_full (the `recommend` scorer) at the same batch size as the
yardstick.

    python scripts/bench_similar_items.py [--k 10] [--out FILE]

Per shape and metric:
  1. mode 0 and mode 1 are checked to return identical ids and score bits on a sample of 64 random queries;
  2. the batch size is chosen among --batches by timing one call of each (CUDA events, after a warm-up call);
  3. the whole job (queries 1..V-1 in fixed-shape batches, tail padded) runs once, timed with CUDA events; re-scored
     candidates per query and queries on the exact fallback are summed over it;
  4. one batch runs under torch.profiler: the share of its kernel time spent in the query-row gather and the table
     normalisation (item_rows_kernel) and in the scorer's operand preparation (pre-split images, item / tile / query
     norms) is reported;
  5. cast_topk_full with random query rows against the raw table at the same batch size (best of 3 calls).
Prints one human line and one JSON line per (shape, metric)."""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import cast_b200  # noqa: E402,F401
from cast_b200 import _lib  # noqa: E402

SHAPES = [("C2", 3417, 50), ("C5", 1000001, 256)]   # (label, V = items + 1, H)
METRICS = {"cosine": 1, "dot": 0}
PREP = ("item_rows_kernel",)                                                    # gather + normalisation
SCORER_PREP = ("presplit_kernel", "item_norm_kernel", "tile_norm_kernel", "tk_unorm_kernel")


def event_ms(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--batches", default="1024,4096,16384")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    K = a.k
    lib = _lib.load_library()
    dev = torch.device("cuda", 0)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                          "0"], capture_output=True, text=True).stdout.strip()
    lines = [f"device: {torch.cuda.get_device_name(0)} | nvidia-smi name, power.limit, clocks.max.sm: {smi}"]
    print(lines[-1], flush=True)
    st = torch.cuda.current_stream().cuda_stream
    for label, V, H in SHAPES:
        g = torch.Generator(device="cpu").manual_seed(0)
        table = (torch.randn(V, H, generator=g) * 0.3).to(dev)
        n_items = V - 1
        for metric, mid in METRICS.items():
            bufs = {}

            def call(q, U, mode, ids, sc, stats, wsb, ws):
                eptr = bufs.setdefault(("eptr", U), torch.arange(U + 1, dtype=torch.int32, device=dev))
                rc = lib.cast_similar_items(q.data_ptr(), U, table.data_ptr(), V, None, 0, V, H, K, mid,
                                            eptr.data_ptr(), q.data_ptr(), mode, ids.data_ptr(), sc.data_ptr(),
                                            None if stats is None else stats.data_ptr(), ws.data_ptr(), wsb, st)
                assert rc == 0, lib.cast_last_error_string()

            def setup(U):
                wsb = lib.cast_similar_items_workspace_bytes(U, V, H, K, mid)
                return (torch.empty(U, K, dtype=torch.int32, device=dev), torch.empty(U, K, device=dev),
                        torch.zeros(2, dtype=torch.int64, device=dev), wsb,
                        torch.empty(wsb // 4 + 16, dtype=torch.int32, device=dev))

            # 1. mode 0 == mode 1 on a sample
            qs = torch.from_numpy(np.random.RandomState(1).choice(np.arange(1, V), 64, replace=False)
                                  .astype(np.int32)).to(dev)
            o0, o1 = setup(64), setup(64)
            call(qs, 64, 0, *o0)
            call(qs, 64, 1, *o1)
            flag = ctypes.c_int(-1)
            lib.cast_similar_items_status(o0[4].data_ptr(), 64, V, H, K, ctypes.byref(flag), st)
            same = bool(torch.equal(o0[0], o1[0]) and torch.equal(o0[1].view(torch.int32), o1[1].view(torch.int32)))
            assert flag.value == 0 and same, ("mode 0 vs mode 1", flag.value, same)
            del o0, o1
            # 2. batch size
            cands = sorted({min(int(b), n_items) for b in a.batches.split(",")})
            per_item = {}
            for B in cands:
                q = torch.arange(1, B + 1, dtype=torch.int32, device=dev)
                o = setup(B)
                call(q, B, 0, *o)
                per_item[B] = event_ms(lambda: call(q, B, 0, *o)) / B
                del o
                torch.cuda.empty_cache()
            B = min(per_item, key=per_item.get)
            # 3. the whole job
            nb = -(-n_items // B)
            qall = torch.ones(nb * B, dtype=torch.int32, device=dev)
            qall[:n_items] = torch.arange(1, V, dtype=torch.int32, device=dev)
            ids, sc, stats, wsb, ws = setup(B)
            tot = torch.zeros(2, dtype=torch.int64, device=dev)
            call(qall[:B], B, 0, ids, sc, stats, wsb, ws)

            def job():
                for b in range(nb):
                    call(qall[b * B:(b + 1) * B], B, 0, ids, sc, stats, wsb, ws)
                    tot.add_(stats)

            job_ms = event_ms(job)
            lib.cast_similar_items_status(ws.data_ptr(), B, V, H, K, ctypes.byref(flag), st)
            assert flag.value == 0, "watchdog"
            rescored, fallback = (int(x) for x in tot.cpu())
            # 4. kernel-time shares of one batch
            from torch.profiler import ProfilerActivity, profile
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                call(qall[:B], B, 0, ids, sc, stats, wsb, ws)
                torch.cuda.synchronize()
            kt = {}
            for e in prof.key_averages():   # kernels and memsets (runtime API entries carry no device time)
                if e.device_time_total > 0 and not e.key.startswith("cuda"):
                    kt[e.key] = kt.get(e.key, 0.0) + e.device_time_total / 1e3
            total_k = sum(kt.values())
            prep = sum(v for k, v in kt.items() if any(p in k for p in PREP))
            sprep = sum(v for k, v in kt.items() if any(p in k for p in SCORER_PREP))
            del ws
            torch.cuda.empty_cache()
            # 5. cast_topk_full at the same U
            users = (torch.randn(B, H, generator=g) * 0.5).to(dev)
            tkb = lib.cast_topk_full_workspace_bytes(B, V, H, K)
            tkw = torch.empty(tkb // 4 + 16, dtype=torch.int32, device=dev)

            def topk():
                rc = lib.cast_topk_full(users.data_ptr(), H, table.data_ptr(), V, H, B, K, None, None, 0,
                                        ids.data_ptr(), sc.data_ptr(), None, tkw.data_ptr(), tkb, st)
                assert rc == 0, lib.cast_last_error_string()

            topk()
            tk_ms = min(event_ms(topk) for _ in range(3))
            del tkw
            torch.cuda.empty_cache()
            batch_ms = job_ms / nb
            r = {"shape": label, "V": V, "H": H, "metric": metric, "K": K, "batch": B, "batches": nb,
                 "job_s": round(job_ms / 1e3, 4), "items_per_s": round(n_items / job_ms * 1e3),
                 "ms_per_batch": round(batch_ms, 4),
                 "candidate_batches_ms_per_1k_items": {b: round(v * 1e3, 4) for b, v in per_item.items()},
                 "rescored_per_query": round(rescored / (nb * B), 1), "fallback_queries": fallback,
                 "profiled_batch_kernel_ms": round(total_k, 4), "gather_normalise_share": round(prep / total_k, 4),
                 "scorer_operand_prep_share": round(sprep / total_k, 4),
                 "topk_full_same_U_ms": round(tk_ms, 4), "ratio_batch_vs_topk_full": round(batch_ms / tk_ms, 3),
                 "mode0_eq_mode1_sample64": same}
            lines.append(f"{label} V={V} H={H} {metric} K={K}: batch {B} ({nb} batches), job {job_ms / 1e3:.3f} s, "
                         f"{n_items / job_ms * 1e3:,.0f} items/s, {batch_ms:.3f} ms/batch | re-scored/query "
                         f"{rescored / (nb * B):.1f}, fallback queries {fallback} | one batch: gather+normalise "
                         f"{100 * prep / total_k:.1f}%, scorer operand prep {100 * sprep / total_k:.1f}% of "
                         f"{total_k:.3f} ms kernel time | cast_topk_full at U={B}: {tk_ms:.3f} ms "
                         f"({batch_ms / tk_ms:.2f}x) | mode0==mode1 on 64 queries {same}")
            print(lines[-1], flush=True)
            lines.append(json.dumps(r))
            print(lines[-1], flush=True)
        del table
        torch.cuda.empty_cache()
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
