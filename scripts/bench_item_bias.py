#!/usr/bin/env python
"""Benchmark of per-item score offsets on exact top-K (cast_topk_full_biased) against the unbiased call, on seeded
random data.

    python scripts/bench_item_bias.py [--reps N] [--rounds R] [--out FILE]

Arms, all on the same users / table / exclusions (50 random items per user):
  unbiased      item_bias = NULL (the kernels of cast_topk_full)
  zero          b = 0 (the biased kernels; same ids and scores as unbiased)
  popularity    b_j = -0.5 log(1 + c_j), c_j seeded Zipf(1.3) counts
  allow90       b_j = 0 for a seeded 90 % of the items, -inf elsewhere
  allow1        the same with 1 %
  allow_lt_k    K / 2 allowed items: fewer than K, so every user takes the exact path
Per (shape, K) every arm is first checked: mode 0 must return the ids and score bits of mode 1 (and zero those of
unbiased), or nothing is timed.  Then, after a warm-up of every arm, the arms are alternated for `rounds` rounds, each
a CUDA-event window of `reps` back-to-back calls; median and spread over the rounds are reported with the candidates
re-scored per user and the users on the exact fallback.  Prints one human line and one JSON line per (shape, K, arm)."""
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
ARMS = ("unbiased", "zero", "popularity", "allow90", "allow1", "allow_lt_k")


def make_bias(arm, V, K, seed=3):
    rng = np.random.RandomState(seed)
    if arm == "unbiased":
        return None
    b = np.zeros(V, np.float32)
    if arm == "popularity":
        b = (-0.5 * np.log1p(rng.zipf(1.3, V).clip(0, 10 ** 7))).astype(np.float32)
    elif arm in ("allow90", "allow1"):
        keep = rng.rand(V) < (0.9 if arm == "allow90" else 0.01)
        b[~keep] = -np.inf
    elif arm == "allow_lt_k":
        b[:] = -np.inf
        b[rng.choice(np.arange(1, V), K // 2, replace=False)] = 0.0
    return b


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    lib = _lib.load_library()
    dev = torch.device("cuda", 0)
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
        for K in KS:
            wsb = lib.cast_topk_full_workspace_bytes(U, V, H, K)
            ws = torch.empty(wsb // 4 + 16, dtype=torch.int32, device=dev)
            ids = [torch.empty(U, K, dtype=torch.int32, device=dev) for _ in range(2)]
            sc = [torch.empty(U, K, dtype=torch.float32, device=dev) for _ in range(2)]
            stats = torch.zeros(2, dtype=torch.int64, device=dev)
            biases = {arm: make_bias(arm, V, K) for arm in ARMS}
            dbias = {arm: None if b is None else torch.from_numpy(b).to(dev) for arm, b in biases.items()}

            def call(arm, mode=0, i=0):
                b = dbias[arm]
                rc = lib.cast_topk_full_biased(users.data_ptr(), H, table.data_ptr(), V, H, U, K, eptr.data_ptr(),
                                               eidx.data_ptr(), None if b is None else b.data_ptr(), mode,
                                               ids[i].data_ptr(), sc[i].data_ptr(), stats.data_ptr(), ws.data_ptr(),
                                               wsb, st)
                assert rc == 0, lib.cast_last_error_string()

            # correctness gate: mode 0 == mode 1 for every arm, zero == unbiased; filter statistics of mode 0
            info, unb = {}, None
            for arm in ARMS:
                call(arm, 1, 1)
                call(arm, 0, 0)
                flag = ctypes.c_int(-1)
                lib.cast_topk_full_status(ws.data_ptr(), U, V, H, K, ctypes.byref(flag), st)
                assert flag.value == 0, "watchdog"
                same = bool(torch.equal(ids[0], ids[1]) and torch.equal(sc[0].view(torch.int32),
                                                                         sc[1].view(torch.int32)))
                assert same, f"{arm}: mode 0 and mode 1 differ"
                if arm == "unbiased":
                    unb = (ids[0].clone(), sc[0].clone())
                if arm == "zero":
                    assert torch.equal(ids[0], unb[0]) and torch.equal(sc[0].view(torch.int32),
                                                                       unb[1].view(torch.int32)), "zero != unbiased"
                rescored, fallback = (int(x) for x in stats.cpu())
                eligible = V - 1 if biases[arm] is None else int(np.isfinite(biases[arm][1:]).sum())
                info[arm] = (rescored / U, fallback, eligible)
            # timing: every arm warmed up, then the arms alternated round by round
            for arm in ARMS:
                call(arm)
                call(arm)
            torch.cuda.synchronize()
            times = {arm: [] for arm in ARMS}
            for _ in range(a.rounds):
                for arm in ARMS:
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    for _ in range(a.reps):
                        call(arm)
                    e1.record()
                    torch.cuda.synchronize()
                    times[arm].append(e0.elapsed_time(e1) / a.reps)
            base = float(np.median(times["unbiased"]))
            for arm in ARMS:
                ms = float(np.median(times[arm]))
                spread = float(max(times[arm]) - min(times[arm]))
                resc, fb, elig = info[arm]
                r = {"shape": label, "U": U, "V": V, "H": H, "K": K, "arm": arm, "ms": round(ms, 4),
                     "spread_ms": round(spread, 4), "vs_unbiased": round(ms / base, 4), "rescored_per_user": round(resc, 1),
                     "fallback_users": fb, "eligible_items": elig, "mode0_eq_mode1": True}
                lines.append(f"{label} U={U} V={V} H={H} K={K} {arm:>10}: {ms:.3f} ms (spread {spread:.3f}) "
                             f"x{ms / base:.3f} of unbiased | re-scored/user {resc:.1f}, fallback users {fb} | "
                             f"eligible items {elig}")
                print(lines[-1], flush=True)
                lines.append(json.dumps(r))
                print(lines[-1], flush=True)
            del ws
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
