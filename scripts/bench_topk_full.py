#!/usr/bin/env python
"""Benchmark of cast_topk_full (exact full-catalog top-K) on random data, with cast_score_rank_full at the same shape
as the yardstick and a torch fp32 mm + topk as context (NOT exact: cuBLAS reorders the sums).

    python scripts/bench_topk_full.py [--reps N] [--out FILE]

Per shape: mode 0 and mode 1 are first checked to return identical ids and score bits, then every call is timed
with CUDA events after warm-up (mean over `reps` back-to-back calls, three windows: median and spread reported).
Every user excludes 50 random items.  Prints one human line and one JSON line per shape."""
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

SHAPES = [  # (label, U, V, H)
    ("C2", 256, 3417, 50),
    ("C5", 256, 1000001, 256),
    ("C5", 2048, 1000001, 256),
]
KS = (10, 100)


def timed(fn, reps, windows=3):
    fn()
    fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(windows):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        out.append(e0.elapsed_time(e1) / reps)
    return float(np.median(out)), float(max(out) - min(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    lib = _lib.load_library()
    dev = torch.device("cuda", 0)
    torch.backends.cuda.matmul.allow_tf32 = False
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                          "0"], capture_output=True, text=True).stdout.strip()
    lines = [f"device: {torch.cuda.get_device_name(0)} | nvidia-smi name, power.limit, clocks.max.sm: {smi}"]
    print(lines[-1], flush=True)
    st = torch.cuda.current_stream().cuda_stream
    for label, U, V, H in SHAPES:
        g = torch.Generator(device="cpu").manual_seed(0)
        table = (torch.randn(V, H, generator=g) * 0.3).to(dev)
        users = (torch.randn(U, H, generator=g) * 0.5).to(dev)
        excl = np.sort(np.random.RandomState(1).randint(1, V, (U, 50)), axis=1).astype(np.int32)
        eptr = torch.arange(0, 50 * (U + 1), 50, dtype=torch.int32, device=dev)
        eidx = torch.from_numpy(excl.reshape(-1)).to(dev)
        # yardstick: full-catalog rank of a random target at the same shape
        target = torch.randint(1, V, (U,), generator=g, dtype=torch.int32).to(dev)
        cgt = torch.zeros(U, dtype=torch.int32, device=dev)
        ceq = torch.zeros_like(cgt)
        sfb = lib.cast_score_rank_full_workspace_bytes(U, V, H)
        sfw = torch.empty(sfb // 4 + 16, dtype=torch.int32, device=dev)

        def score_full():
            rc = lib.cast_score_rank_full(users.data_ptr(), H, table.data_ptr(), V, H, U, target.data_ptr(), None,
                                          None, None, 0, cgt.data_ptr(), ceq.data_ptr(), None, sfw.data_ptr(), sfb, st)
            assert rc == 0, lib.cast_last_error_string()

        sf_ms, sf_spread = timed(score_full, a.reps)
        del sfw
        for K in KS:
            ids = [torch.empty(U, K, dtype=torch.int32, device=dev) for _ in range(2)]
            sc = [torch.empty(U, K, dtype=torch.float32, device=dev) for _ in range(2)]
            stats = torch.zeros(2, dtype=torch.int64, device=dev)
            wsb = lib.cast_topk_full_workspace_bytes(U, V, H, K)
            ws = torch.empty(wsb // 4 + 16, dtype=torch.int32, device=dev)

            def topk(mode, i=0):
                rc = lib.cast_topk_full(users.data_ptr(), H, table.data_ptr(), V, H, U, K, eptr.data_ptr(),
                                        eidx.data_ptr(), mode, ids[i].data_ptr(), sc[i].data_ptr(), stats.data_ptr(),
                                        ws.data_ptr(), wsb, st)
                assert rc == 0, lib.cast_last_error_string()

            topk(1, 1)
            topk(0, 0)
            flag = ctypes.c_int(-1)
            lib.cast_topk_full_status(ws.data_ptr(), U, V, H, K, ctypes.byref(flag), st)
            assert flag.value == 0, "watchdog"
            same = bool(torch.equal(ids[0], ids[1]) and torch.equal(sc[0].view(torch.int32), sc[1].view(torch.int32)))
            assert same, "mode 0 and mode 1 differ"
            rescored, fallback = (int(x) for x in stats.cpu())
            ms, spread = timed(lambda: topk(0), a.reps)
            del ws

            def ref():   # context only: fp32 logits materialised, reordered sums
                s = users @ table.T
                s[:, 0] = -float("inf")
                s.scatter_(1, eidx.view(U, 50).long(), -float("inf"))
                return torch.topk(s, K, dim=1)

            mm_ms, _ = timed(ref, a.reps)
            r = {"shape": label, "U": U, "V": V, "H": H, "K": K, "ms": round(ms, 4), "spread_ms": round(spread, 4),
                 "users_per_s": round(U / ms * 1e3), "score_rank_full_ms": round(sf_ms, 4),
                 "ratio_vs_score_rank_full": round(sf_ms / ms, 3), "rescored_per_user": round(rescored / U, 1),
                 "fallback_users": fallback, "mode0_eq_mode1": same, "torch_mm_topk_nonexact_ms": round(mm_ms, 4),
                 "table_in_l2": V * H * 4 < 126e6}
            lines.append(f"{label} U={U} V={V} H={H} K={K}: {ms:.3f} ms (spread {spread:.3f}) {U / ms * 1e3:,.0f} users/s"
                         f" | score_rank_full {sf_ms:.3f} ms -> ratio {sf_ms / ms:.2f}x | re-scored/user "
                         f"{rescored / U:.1f}, fallback users {fallback} | mode0==mode1 {same} | torch fp32 mm+topk "
                         f"(non-exact) {mm_ms:.3f} ms" + (" | table in L2" if r["table_in_l2"] else ""))
            print(lines[-1], flush=True)
            lines.append(json.dumps(r))
            print(lines[-1], flush=True)
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
