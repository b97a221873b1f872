#!/usr/bin/env python
"""Per-kernel GPU time of the three attention kernels (forward, dQ, dK/dV) in the bench's training step: the bench's
model and synthetic batches (`--config`, default c2), eager launches (no graph) so that every kernel is its own
profiler event, `--steps` steps under torch.profiler after `--warmup`.  Prints one line per kernel: launches per step,
mean and total microseconds per step.  `--root` selects the source tree whose built library is imported (a second
checkout, for parent-vs-new comparisons).

    python scripts/bench_attention_kernels.py [--root DIR] [--config c2] [--steps 50] [--warmup 10]
"""
import argparse
import os
import sys
from collections import defaultdict

ap = argparse.ArgumentParser()
ap.add_argument("--root", default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
ap.add_argument("--config", default="c2")
ap.add_argument("--steps", type=int, default=50)
ap.add_argument("--warmup", type=int, default=10)
a = ap.parse_args()
sys.path.insert(0, os.path.abspath(a.root))

import torch  # noqa: E402
from torch.profiler import ProfilerActivity, profile  # noqa: E402

import bench  # noqa: E402
import cast_b200  # noqa: E402

bench.select_config(a.config)
dev = torch.device("cuda", 0)
torch.cuda.set_device(dev)
args = bench.make_args(128)
model = cast_b200.build_model(bench.CFG["model"], bench.USERNUM, bench.ITEMNUM, 5, args, device=dev, use_graph=False)
batches = bench.synth_batches(8, 128, args.maxlen, bench.ITEMNUM, seed=20191019)
for i in range(a.warmup):
    model.train_step(None, *batches[i % len(batches)])
torch.cuda.synchronize()
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for i in range(a.steps):
        model.train_step(None, *batches[i % len(batches)])
    torch.cuda.synchronize()
agg = defaultdict(lambda: [0, 0.0])
for e in prof.events():
    if e.device_type == torch.autograd.DeviceType.CUDA and "attn_" in e.name:
        name = e.name.split("(")[0].replace("void ", "")
        agg[name][0] += 1
        agg[name][1] += e.time_range.elapsed_us()
print(f"{torch.cuda.get_device_name(0)}, config {a.config}, {a.steps} steps, tree {os.path.basename(os.path.abspath(a.root))}")
for name, (n, us) in sorted(agg.items()):
    print(f"  {name:60s} {n / a.steps:4.1f}/step  mean {us / n:7.2f} us  {us / a.steps:7.2f} us/step")
