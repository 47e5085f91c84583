#!/usr/bin/env python
"""Per-step time curve of the AR stacks (VERDICT r1 item 5c): one reference-faithful step of MegaPLM.infer / MegaADM.infer at
sequence length S = t + 1 is one non-causal pass of the stack over (B, S, D) with the last layer pruned to its last row
(csrc/drivers.cu encoder_forward, last_row_only).  Prints per S: ms per step, algorithmic dense-layer + attention FLOPs, the
achieved fp32-equivalent TFLOP/s and launches per step.  GPU only; eager launches (the product replays the same sequence from
a CUDA graph).

    python tools/ar_step_curve.py [--batch 64] [--steps 1 2 4 8 12 16 24 32 48 64]
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import helpers  # noqa: E402
from oracle import weights  # noqa: E402  (seeded weight specs only; nothing of the oracle is timed)
from megatts2_b200 import ops  # noqa: E402
from megatts2_b200.modules.transformer import run_encoder  # noqa: E402

DEV = "cuda:0"


def step_flops(B, S, D, F, n_layers):
    """dense layers (QKV, out-proj, FF1, FF2) + attention (QK^T, PV) of one pass; the last layer's out-proj / FFN / query
    side only for the last row (the exact pruning the driver takes)."""
    full = 2.0 * B * S * (3 * D * D + D * D + 2 * D * F) + 4.0 * B * S * S * D
    last = 2.0 * B * S * (3 * D * D) + 2.0 * B * (D * D + 2 * D * F) + 4.0 * B * S * D
    return (n_layers - 1) * full + last


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--steps", type=int, nargs="*", default=[1, 2, 3, 4, 6, 8, 12, 16, 24, 32, 48, 64])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--quiet", action="store_true", help="totals only")
    ap.add_argument("--infer", action="store_true", help="also time the graph-replayed MegaPLM.infer / MegaADM.infer (T = 64)")
    a = ap.parse_args()
    plm = helpers.build_plm(weights.plm_state_dict(), DEV)
    adm = helpers.build_adm(weights.adm_state_dict(), DEV)
    g = torch.Generator().manual_seed(11)
    for name, enc in (("plm", plm.plm), ("adm", adm.adm)):
        layers = list(enc.layers)
        D, FF, n = layers[0].dim, layers[0].ff_dim, len(layers)
        tot_ms = 0.0
        per_s = {}
        for S in a.steps:
            x = torch.randn(a.batch, S, D, generator=g).to(DEV)
            for _ in range(2):
                run_encoder(enc, layers, x, None, last_row_only=True)
            torch.cuda.synchronize()
            n0 = ops.launch_count()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(a.reps):
                run_encoder(enc, layers, x, None, last_row_only=True)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / a.reps
            fl = step_flops(a.batch, S, D, FF, n)
            tot_ms += ms
            per_s[S] = ms
            if a.quiet:
                continue
            print(json.dumps({"stack": name, "B": a.batch, "S": S, "rows": a.batch * S, "ms_per_step": round(ms, 3),
                              "gflop": round(fl / 1e9, 1), "tflops_fp32_equiv": round(fl / ms / 1e9, 1),
                              "launches": (ops.launch_count() - n0) // a.reps}), flush=True)
        row = {"stack": name, "sum_ms_over_listed_steps": round(tot_ms, 2), "steps": len(a.steps)}
        if a.infer:
            tc = torch.relu(torch.randn(a.batch, 64, 512, generator=g)).to(DEV)
            row["infer_T64_ms"] = timed_infer((plm if name == "plm" else adm).infer, tc)
        print(json.dumps(row), flush=True)


def timed_infer(fn, x, n=7):
    ms = []
    for _ in range(n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn(x)
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    return round(min(ms[3:]), 2)


if __name__ == "__main__":
    main()
