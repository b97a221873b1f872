"""Step time of global-norm gradient clipping (args.clip_grad), one GPU, same process.

Three arms per optimizer ("adam", "lazy_adam"): clipping off; on with max_norm = 1e30 (norm and scale computed, never
clips); on with max_norm = 1e-6 (clips every step).  The models are built from bench.py's CONFIGS / synth_batches (the
same seeded batches); steps are graph replays with per-step CUDA events and the L2 flushed (256 MiB write) before every
step, as bench.py does.  The arms alternate round by round in a rotating order so drift of the shared machine lands on
all of them; the result is the median over rounds of the per-round median, with the spread (max - min) of the rounds.
Also printed: the distribution of the pre-clip global norm over the seeded batches under the default max_norm 5.0 (a
fresh model trained for --norm_steps steps with clipping at 5.0), i.e. whether the default ever clips at these shapes.

  python scripts/bench_grad_clip.py [--configs c2,c5] [--rounds 4] [--steps 40] [--warmup 5] [--out FILE]
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

ARMS = {"off": {}, "on_no_clip": {"clip_grad": True, "max_norm": 1e30},
        "on_clipping": {"clip_grad": True, "max_norm": 1e-6}}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else torch.cuda.get_device_name(0)


def build(cfg_batches, B, opt, dev, **kw):
    import cast_b200
    args = bench.make_args(B)
    args.optimizer = opt
    for k, v in kw.items():
        setattr(args, k, v)
    m = cast_b200.build_model(bench.CFG["model"], bench.USERNUM, bench.ITEMNUM, 5, args, device=dev, use_graph=True)
    m.train_step(None, *cfg_batches[0])          # buffers + graph capture
    return m


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="c2,c5")
    ap.add_argument("--optimizers", default="adam,lazy_adam")
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--norm_steps", type=int, default=64)
    ap.add_argument("--batch_size", type=int, default=128)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    lines = [f"card (name, power.limit, clocks.max.sm): {card()}"]
    print(lines[0], flush=True)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    for cfg in a.configs.split(","):
        bench.select_config(cfg)
        B = a.batch_size
        batches = bench.synth_batches(8, B, bench.CFG["T"], bench.ITEMNUM, seed=20191019)
        dev_batches = [(torch.from_numpy(np.stack([x.reshape(-1) for x in b[:3]])).to(dev),
                        torch.from_numpy(np.stack([x.reshape(-1) for x in b[3:]])).to(dev)) for b in batches]
        for opt in a.optimizers.split(","):
            models = {arm: build(batches, B, opt, dev, **kw) for arm, kw in ARMS.items()}
            names = list(models)
            times = {arm: [] for arm in models}
            for r in range(a.rounds):
                order = names[r % len(names):] + names[:r % len(names)]
                for arm in order:
                    m = models[arm]
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
                    times[arm].append(float(np.median([e0.elapsed_time(e1) for e0, e1 in ev])))
            res = {"config": cfg, "optimizer": opt, "workload": bench.CFG["desc"], "batch": B,
                   "n_params": models["off"].engine.n_params}
            for arm in models:
                t = times[arm]
                res[arm] = {"ms_per_step_median_per_round": [round(x, 4) for x in t],
                            "ms_per_step": round(float(np.median(t)), 4), "spread_ms": round(max(t) - min(t), 4),
                            "launches_per_step": models[arm].launches_per_step}
            for arm in ("on_no_clip", "on_clipping"):
                res[arm]["added_ms"] = round(res[arm]["ms_per_step"] - res["off"]["ms_per_step"], 4)
            del models
            torch.cuda.empty_cache()
            # pre-clip norms under the default threshold
            m = build(batches, B, opt, dev, clip_grad=True, max_norm=5.0)
            norms = []
            for i in range(a.norm_steps):
                m.train_step(None, *batches[(i + 1) % len(batches)])
                norms.append(m.last_grad_norm())
            q = np.quantile(norms, [0.0, 0.1, 0.5, 0.9, 1.0])
            res["grad_norm_at_default_max_norm_5"] = {
                "steps": a.norm_steps, "min": round(float(q[0]), 5), "p10": round(float(q[1]), 5),
                "median": round(float(q[2]), 5), "p90": round(float(q[3]), 5), "max": round(float(q[4]), 5),
                "first": round(float(norms[0]), 5), "steps_clipped": int(sum(x > 5.0 for x in norms))}
            del m
            torch.cuda.empty_cache()
            lines.append(json.dumps(res))
            print(lines[-1], flush=True)
    lines.append(f"card (name, power.limit, clocks.max.sm): {card()}")
    print(lines[-1])
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
