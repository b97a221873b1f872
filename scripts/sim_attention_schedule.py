#!/usr/bin/env python
"""Replay the launch order of the attention kernels on the bench's synthetic C2 batches: how many (sequence, 64-row
tile) CTAs are live, how much work each has, and how long the kernel must last on 148 SMs x 2 resident CTAs when a
CTA cannot be split — the explanation of the idle SM-time ncu reports (DESIGN.md 4c).  CPU only.

Work is counted in staged chunks: 64-key chunks for the forward and dQ kernels (per query tile), 32-query chunks for
the dK/dV kernel (per key tile).  Per-CTA overheads are ignored.  The block scheduler is modelled as a greedy fill:
each CTA, in grid order, goes to the slot that frees first.  Rows and keys start at the first kept key (left padding;
the training step passes skip_ids, so there are no uniform rows).

  fwd/dQ: as launched (last query tile first); the same rows as 32-row tiles on four resident CTAs per SM (a slot
          of that configuration runs at half the speed); and an adaptive split (a tile of >= --fwd-min chunks runs
          as two 32-row halves, each at half the cost per chunk: four key groups of 16 keys instead of two of 32);
  dK/dV:  last key tile first (the order before the key-tile map), heaviest first (first key tile first, as the
          kernel launches now), and an adaptive split (a key tile needing >= --dkv-min query chunks runs as two
          32-key halves, each warp taking one 8-query k-step of every chunk instead of two).
Light tiles' second slots exit at once and cost nothing here.  The model favours the splits; on the GPU they were
slower (DESIGN.md 4c): a CTA's chunk costs its staging latency and barriers as much as its arithmetic, which the
model leaves out.

    python scripts/sim_attention_schedule.py [--fwd-min 3] [--dkv-min 4] [--sweep]
"""
import argparse
import heapq
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from bench import synth_batches  # noqa: E402

B, T, TILE, CH, TQ, SLOTS = 128, 200, 64, 64, 32, 296
ntile = (T + TILE - 1) // TILE
nqch = (T + TQ - 1) // TQ


def makespan(tasks, nslots=SLOTS):
    slots = [0.0] * nslots
    heapq.heapify(slots)
    for n in tasks:
        heapq.heappush(slots, heapq.heappop(slots) + n)
    return max(slots), sum(tasks) / nslots


def fwd_chunks(first, q0, w):
    """64-key chunks of the query rows q0..q0+w-1 (attn_fwd_mma_kernel / attn_bwd_dq_mma_kernel: kbeg..kend)."""
    if q0 + w <= first:
        return 0
    kbeg = (first // CH) * CH
    return (q0 + w - kbeg + CH - 1) // CH


def dkv_chunks(first, k0):
    """32-query chunks (aligned to the end of the sequence) that reach keys >= k0 (attn_bwd_dkv_ws_kernel: needed)."""
    n = 0
    for cc in range(nqch):
        c0 = T - (nqch - cc) * TQ
        if c0 + TQ > first and c0 + TQ > k0:
            n += 1
    return n


def tasks_fwd(firsts, split_min):
    out = []
    for tile in reversed(range(ntile)):          # grid order: last (heaviest) query tile first
        q0 = T - TILE * (ntile - tile)
        for f in firsts:
            n = fwd_chunks(f, q0, TILE)
            if n == 0:
                continue                          # padding-only tile: exits at once
            if split_min and n >= split_min:
                out += [0.5 * fwd_chunks(f, q0 + 32 * s, 32) for s in range(2)]
            else:
                out.append(n)
    return out


def tasks_dkv(firsts, order, split_min):
    out = []
    tiles = range(ntile) if order == "first" else reversed(range(ntile))
    for tile in tiles:
        k0 = T - TILE * (ntile - tile)
        for f in firsts:
            if k0 + TILE <= f:
                continue                          # keys all before the sequence: zero gradient, exits at once
            n = dkv_chunks(f, k0)
            if split_min and n >= split_min:
                out += [0.5 * dkv_chunks(f, k0 + 32 * s) for s in range(2)]
            else:
                out.append(n)
    return out


def fmt(tasks):
    mk, per = makespan(tasks)
    return f"makespan {mk:4.1f} (ideal {per:4.2f}, efficiency {per / mk:.2f})"


ap = argparse.ArgumentParser()
ap.add_argument("--fwd-min", type=int, default=3)
ap.add_argument("--dkv-min", type=int, default=4)
ap.add_argument("--sweep", action="store_true", help="mean makespan over the batches for every threshold")
a = ap.parse_args()
batches = [T - (b[0] != 0).sum(1) for b in synth_batches(4, B, T, 3416, seed=20191019)]
for bi, firsts in enumerate(batches):
    L = T - firsts
    print(f"batch {bi}: mean length {L.mean():.0f}, full-length {np.mean(L == T):.2f}")
    tasks = tasks_fwd(firsts, 0)
    print(f"  fwd/dQ  as launched      {fmt(tasks)}: {len(tasks)} live tiles of {B * ntile}, heaviest {max(tasks)}")
    fine = []
    nt32 = (T + 31) // 32
    for tile in reversed(range(nt32)):
        for f in firsts:
            n = fwd_chunks(f, T - 32 * (nt32 - tile), 32)
            if n:
                fine.append(0.5 * n)
    mk4 = 2 * makespan(fine, 2 * SLOTS)[0]
    print(f"  fwd/dQ  32-row tiles, 4 CTAs/SM: makespan {mk4:4.1f} (efficiency {sum(fine) / SLOTS / mk4:.2f})")
    print(f"  fwd/dQ  split >= {a.fwd_min}      {fmt(tasks_fwd(firsts, a.fwd_min))}")
    print(f"  dK/dV   last tile first  {fmt(tasks_dkv(firsts, 'last', 0))}")
    print(f"  dK/dV   heaviest first   {fmt(tasks_dkv(firsts, 'first', 0))}")
    print(f"  dK/dV   split >= {a.dkv_min}      {fmt(tasks_dkv(firsts, 'first', a.dkv_min))}")
if a.sweep:
    for m in range(1, 8):
        fw = np.mean([makespan(tasks_fwd(f, m))[0] for f in batches])
        dk = np.mean([makespan(tasks_dkv(f, "first", m))[0] for f in batches])
        print(f"threshold {m}: mean makespan fwd/dQ {fw:.2f}, dK/dV {dk:.2f}")
