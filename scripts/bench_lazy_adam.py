"""Step time of optimizer="adam" (dense TF-Adam) vs "lazy_adam" (LazyAdam on the item table), one GPU, same process.

Both models are built from bench.py's CONFIGS / synth_batches (the same seeded batches), steps are graph replays with
per-step CUDA events and the L2 flushed (256 MiB write) before every step, as bench.py does.  The two optimizers
alternate round by round (A B, B A, ...) so drift of the shared machine lands on both.  Also printed: the eager
optimizer segment (the Adam launches, plus the embedding-gradient scatters whose zeroing pass lazy_adam drops) timed
with per-launch events, and the distinct item ids the batches touch.

  python scripts/bench_lazy_adam.py [--configs c5,c2] [--rounds 4] [--steps 40] [--warmup 5] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else torch.cuda.get_device_name(0)


def segment_ms(model, c):
    """eager per-launch events of one step: (Adam launches, embedding-gradient scatters incl. sort and zeroing) in ms"""
    eng = model.engine
    eng.timing = []
    eng.launch_train_step(c)
    torch.cuda.synchronize()
    adam = sum(e0.elapsed_time(e1) for n, _, e0, e1 in eng.timing if n.startswith("cast_adam"))
    scat = sum(e0.elapsed_time(e1) for n, _, e0, e1 in eng.timing if n.startswith("cast_scatter"))
    eng.timing = None
    return adam, scat


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="c5,c2")
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch_size", type=int, default=128)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import cast_b200
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    lines = [f"card (name, power.limit, clocks.max.sm): {card()}"]
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    for cfg in a.configs.split(","):
        bench.select_config(cfg)
        B = a.batch_size
        batches = bench.synth_batches(8, B, bench.CFG["T"], bench.ITEMNUM, seed=20191019)
        touched = [len(np.unique(np.concatenate([x.reshape(-1) for x in b[:3]]))) - 1 for b in batches]
        dev_batches = [(torch.from_numpy(np.stack([x.reshape(-1) for x in b[:3]])).to(dev),
                        torch.from_numpy(np.stack([x.reshape(-1) for x in b[3:]])).to(dev)) for b in batches]
        models = {}
        for opt in ("adam", "lazy_adam"):
            args = bench.make_args(B)
            args.optimizer = opt
            m = cast_b200.build_model(bench.CFG["model"], bench.USERNUM, bench.ITEMNUM, 5, args, device=dev,
                                      use_graph=True)
            m.train_step(None, *batches[0])          # buffers + graph capture
            models[opt] = m
        times = {opt: [] for opt in models}
        for r in range(a.rounds):
            order = ("adam", "lazy_adam") if r % 2 == 0 else ("lazy_adam", "adam")
            for opt in order:
                m = models[opt]
                c = m.engine.ctx(B)
                ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
                      for _ in range(a.steps)]
                for i in range(a.warmup + a.steps):
                    k3, c3 = dev_batches[i % len(dev_batches)]
                    c.keys3.copy_(k3)
                    c.cids.copy_(c3)
                    if i >= a.warmup:
                        flush.zero_()
                        ev[i - a.warmup][0].record()
                    m.launch(c)
                    if i >= a.warmup:
                        ev[i - a.warmup][1].record()
                torch.cuda.synchronize()
                times[opt].append(float(np.median([e0.elapsed_time(e1) for e0, e1 in ev])))
        seg = {}
        for opt, m in models.items():
            c = m.engine.ctx(B)
            c.keys3.copy_(dev_batches[1][0])
            c.cids.copy_(dev_batches[1][1])
            seg[opt] = [segment_ms(m, c) for _ in range(5)][1:]
        res = {"config": cfg, "workload": bench.CFG["desc"], "batch": B,
               "touched_rows_per_step": {"mean": float(np.mean(touched)), "min": int(min(touched)),
                                         "max": int(max(touched)), "table_rows": bench.ITEMNUM + 1}}
        for opt in models:
            t = times[opt]
            res[opt] = {"ms_per_step_median_per_round": [round(x, 4) for x in t],
                        "ms_per_step": round(float(np.median(t)), 4),
                        "spread_ms": round(max(t) - min(t), 4),
                        "eager_adam_ms": round(float(np.median([s[0] for s in seg[opt]])), 4),
                        "eager_scatter_ms": round(float(np.median([s[1] for s in seg[opt]])), 4)}
        res["speedup"] = round(res["adam"]["ms_per_step"] / res["lazy_adam"]["ms_per_step"], 4)
        lines.append(json.dumps(res))
        print(lines[-1], flush=True)
        del models
        torch.cuda.empty_cache()
    lines.append(f"card (name, power.limit, clocks.max.sm): {card()}")
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")
    print(lines[0])


if __name__ == "__main__":
    main()
