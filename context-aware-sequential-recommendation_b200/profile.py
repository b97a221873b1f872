"""Per-kernel timing of one training step with CUDA events on the launch stream, and the roofline arithmetic for the
dominant kernel (algorithmic FLOPs / bytes from the call's own arguments; peaks from MEASURED_PEAKS.json)."""
from __future__ import annotations

import json
import os
from collections import defaultdict

import torch

FALLBACK_PEAKS = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}


def _work(name, a, B, T, H, h):
    """(flops, hbm_bytes) algorithmic work of one C-ABI call, derived from its arguments (include/cast_b200.h)."""
    if name == "cast_gemm":
        M, N, K = a[8], a[9], a[10]
        return 2.0 * M * N * K, 4.0 * (M * K + K * N + M * N)
    if name == "cast_attn_fwd":   # dense T x T: QK^T + PV  (SURVEY §8d "4TH per row")
        return 4.0 * B * T * T * H, 4.0 * 5 * B * T * H
    if name == "cast_attn_bwd":   # dP, dQ, dK, dV = 2x forward (algorithmic; recomputation of S not counted)
        return 8.0 * B * T * T * H, 4.0 * 8 * B * T * H
    if name == "cast_rowk_ln_qkv_fwd":  # 3 projections  (a[7]=N, a[8]=H)
        return 6.0 * a[7] * a[8] * a[8], 4.0 * 5 * a[7] * a[8]
    if name == "cast_rowk_ln_ffn_fwd":  # 2 GEMMs        (a[12]=N, a[13]=H)
        return 4.0 * a[12] * a[13] * a[13], 4.0 * 4 * a[12] * a[13]
    if name == "cast_ffn_bwd":      # 2 dgrad + 2 wgrad  (a[14]=N, a[15]=H)
        return 8.0 * a[14] * a[15] * a[15], 4.0 * 5 * a[14] * a[15]
    if name in ("cast_qkv_bwd", "cast_qkv_bwd_embed"):      # 3 dgrad + 3 wgrad  (a[12]=N, a[13]=H in both forms)
        return 12.0 * a[12] * a[13] * a[13], 4.0 * 7 * a[12] * a[13]
    if name in ("cast_layernorm_fwd",):
        return 8.0 * a[3] * a[4], 4.0 * 2 * a[3] * a[4]
    if name in ("cast_layernorm_bwd",):
        return 12.0 * a[5] * a[6], 4.0 * 3 * a[5] * a[6]
    if name == "cast_embed_fwd":
        return 3.0 * a[4] * a[3], 4.0 * (2 * a[4] * a[3] + a[4])
    if name == "cast_mask_dropout":
        return 2.0 * a[6] * a[7], 4.0 * 3 * a[6] * a[7]
    if name == "cast_adam_tf_step":
        return 12.0 * a[4], 28.0 * a[4]
    if name == "cast_logits_loss":
        return 6.0 * a[4] * a[3], 4.0 * 4 * a[4] * a[3]
    if name == "cast_lnf_loss":     # LN + 2 gathers + dots + LN backward: x, 2 table rows in; seq_emb, dx out (a[6]=H, a[7]=N)
        return 30.0 * a[7] * a[6], 4.0 * 5 * a[7] * a[6]
    if name == "cast_scatter_rows":
        n, nsrc, Hh, V = a[2], a[1], a[7], a[6]
        return 2.0 * n * nsrc * Hh, 4.0 * (n * nsrc * Hh + V * Hh) + 16.0 * n * nsrc
    if name == "cast_colsum":
        return 1.0 * a[1] * a[2], 4.0 * a[1] * a[2]
    return 0.0, 0.0


def profile_step(model, c, steps=5):
    """Runs `steps` eager training steps with every C-ABI call bracketed by CUDA events; returns a list of
    {name, calls_per_step, ms_per_step, share, tflops, gbs} sorted by time."""
    eng = model.engine
    B, T, H, h = c.B, eng.T, eng.H, eng.h
    with eng.rank_local():      # rank-local profiling: no barrier, exchange or peer read in here
        eng.launch_train_step(c)  # warm
        torch.cuda.synchronize(eng.device)
        eng.timing = []
        try:
            for _ in range(steps):
                eng.launch_train_step(c)
            torch.cuda.synchronize(eng.device)
        finally:
            rec, eng.timing = eng.timing, None
    agg = defaultdict(lambda: [0, 0.0, 0.0, 0.0])
    for name, a, e0, e1 in rec:
        ms = e0.elapsed_time(e1)
        fl, by = _work(name, a, B, T, H, h)
        r = agg[name]
        r[0] += 1
        r[1] += ms
        r[2] += fl
        r[3] += by
    total = sum(r[1] for r in agg.values()) or 1.0
    out = []
    for name, (n, ms, fl, by) in agg.items():
        out.append({"name": name, "calls_per_step": n / steps, "ms_per_step": ms / steps, "share": ms / total,
                    "tflops": fl / (ms * 1e-3) / 1e12 if ms > 0 else 0.0,
                    "gbs": by / (ms * 1e-3) / 1e9 if ms > 0 else 0.0,
                    "flops_per_step": fl / steps, "bytes_per_step": by / steps})
    out.sort(key=lambda r: -r["ms_per_step"])
    return out


def load_peaks(root):
    p = os.path.join(root, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        with open(p) as f:
            d = json.load(f)
        d["source"] = "measured"
        return d
    d = dict(FALLBACK_PEAKS)
    d["source"] = "fallback"
    return d


COMPUTE_BOUND = ("cast_attn_fwd", "cast_attn_bwd", "cast_gemm", "cast_qkv_bwd", "cast_qkv_bwd_embed", "cast_ffn_bwd",
                 "cast_rowk_ln_qkv_fwd", "cast_rowk_ln_ffn_fwd")


def ncu_traffic(root, name):
    """DRAM bytes per launch of a C-ABI call from the committed ncu `--set full` capture (profiles/traffic.json:
    {call: {"dram_bytes": read+write summed over the call's kernels, "source": file}}), or None."""
    p = os.path.join(root, "profiles", "traffic.json")
    if not os.path.isfile(p):
        return None, None
    with open(p) as f:
        d = json.load(f)
    e = d.get(name)
    return (e["dram_bytes"], e.get("source")) if e else (None, None)


def roofline_of_dominant(kernels, B, T, H, args, root):
    if not kernels:
        return None
    top = kernels[0]
    pk = load_peaks(root)
    traffic, tsrc = ncu_traffic(root, top["name"])
    if top["name"] in COMPUTE_BOUND:
        peak = pk.get("bf16_tflops_sustained", pk["bf16_tflops"])
        fp32_peak = 2 * 128 * 148 * pk.get("sm_max_mhz", 1965.0) * 1e6 / 1e12
        # fp32-grade results need the 3xTF32 split: 3 tensor passes per algorithmic product, at half the bf16 rate
        eff_peak = peak / 2.0 / 3.0
        mma_peak = 1024 * 148 * pk.get("sm_max_mhz", 1965.0) * 1e6 / 1e12
        narrow = H <= 64 and top["name"] != "cast_gemm"
        pipe = ("tensor cores, mma.sync m16n8k8 TF32 x3 (hi/lo split keeps fp32 parity 1e-4); head width "
                f"{H} < one UMMA tile, so warp-level MMA with register-resident softmax"
                if narrow else "tensor cores, tcgen05.mma kind::tf32 x3 (3xTF32 split, TMEM accumulators)")
        return {"kernel": top["name"], "bound": "tensor", "achieved": top["tflops"], "peak": peak, "unit": "TFLOP/s",
                "frac": top["tflops"] / peak, "traffic": traffic, "traffic_source": tsrc,
                "peak_source": pk["source"] + " (sustained bf16 cuBLAS)",
                "share_of_step": top["share"], "ms_per_step": top["ms_per_step"],
                "algorithmic_flops_per_step": top["flops_per_step"],
                "pipe_used": pipe,
                "peak_3xtf32_tflops": eff_peak, "frac_of_3xtf32_peak": top["tflops"] / eff_peak,
                # warp-level path: HMMA.1688.F32.TF32 holds the SMSP tensor pipe 8 cycles (measured, ncu:
                # pipe_tensor_cycles_active / HMMA count, profiles/r02_mma_sync_rate.txt) => 1024 flop/clk/SM
                "mma_sync_tf32_peak_tflops": mma_peak, "frac_of_mma_sync_3xtf32": top["tflops"] / (mma_peak / 3.0),
                "fp32_pipe_peak_tflops": fp32_peak, "frac_of_fp32_pipe": top["tflops"] / fp32_peak}
    peak = pk["hbm_gbs"]
    return {"kernel": top["name"], "bound": "hbm", "achieved": top["gbs"], "peak": peak, "unit": "GB/s",
            "frac": top["gbs"] / peak, "traffic": traffic, "traffic_source": tsrc, "peak_source": pk["source"],
            "share_of_step": top["share"],
            "ms_per_step": top["ms_per_step"], "algorithmic_bytes_per_step": top["bytes_per_step"]}
