"""Per-shape throughput of the tensor-core tap-GEMM with the launch plan the dispatcher picks (diagnostics, GPU only).

For each shape runs the op `reps` times inside the library's event trace and reports the main kernel's
time per launch (the activation split is traced separately) and its rate in fp32-equivalent TFLOP/s
(2*M*N*K*k; the tensor pipe executes 6 bf16 MMAs per fp32 product, so dense-bf16-equivalent = 6x).
"""
import ctypes as C
import math
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from megatts2_b200 import _lib as L, ops, pack  # noqa: E402

DEV = "cuda:0"
SHAPES = [
    # PLM / ADM dense layers (k = 1): rows = batch x sequence
    dict(name="plm qkv  M5888 K1024 N3072", B=1, T=5888, Cin=1024, Cout=3072, k=1),
    dict(name="plm ff1  M5888 K1024 N4096", B=1, T=5888, Cin=1024, Cout=4096, k=1),
    dict(name="plm ff2  M5888 K4096 N1024", B=1, T=5888, Cin=4096, Cout=1024, k=1),
    dict(name="plm out  M5888 K1024 N1024", B=1, T=5888, Cin=1024, Cout=1024, k=1),
    # HiFi-GAN ResBlock convs
    dict(name="hifi s1  C256 k7  T4176 B64", B=64, T=4176, Cin=256, Cout=256, k=7, dil=3),
    dict(name="hifi s2  C128 k7  T8352 B64", B=64, T=8352, Cin=128, Cout=128, k=7, dil=3),
    dict(name="hifi s3  C64  k7  T33408 B64", B=64, T=33408, Cin=64, Cout=64, k=7, dil=3),
    dict(name="hifi s4  C32  k7  T66816 B64", B=64, T=66816, Cin=32, Cout=32, k=7, dil=3),
    # AR-loop shapes at smaller steps (rows = 64 x t)
    dict(name="plm ff1  M2048 K1024 N4096", B=1, T=2048, Cin=1024, Cout=4096, k=1),
    dict(name="plm ff2  M2048 K4096 N1024", B=1, T=2048, Cin=4096, Cout=1024, k=1),
    dict(name="plm qkv  M1024 K1024 N3072", B=1, T=1024, Cin=1024, Cout=3072, k=1),
    dict(name="adm qkv  M4096 K768  N2304", B=1, T=4096, Cin=768, Cout=2304, k=1),
    dict(name="adm ff1  M4096 K768  N1024", B=1, T=4096, Cin=768, Cout=1024, k=1),
]


def trace_ms(fn, reps):
    lib = L.lib()
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    lib.mtts_trace_begin(ops._stream())
    for _ in range(reps):
        fn()
    buf = C.create_string_buffer(16384)
    lib.mtts_trace_end(buf, 16384)
    for line in buf.value.decode().splitlines():
        f = line.split()
        if f and f[0] == "conv_tc_launch":
            return float(f[2]) / int(f[1])
    return float("nan")


def main():
    import argparse
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--shapes", type=str, default="", help="comma-separated shape indices (default: all)")
    ap.add_argument("--fmt", type=str, default="f16x2", choices=["f16x2", "bf16x3"])
    args = ap.parse_args()
    reps = args.reps
    shapes = [SHAPES[int(i)] for i in args.shapes.split(",")] if args.shapes else SHAPES
    g = torch.Generator().manual_seed(0)
    for s in shapes:
        k, dil = s["k"], s.get("dil", 1)
        pad = dil * (k - 1) // 2
        x = torch.randn(s["B"], s["T"], s["Cin"], generator=g).to(DEV)
        w = torch.randn(s["Cout"], s["Cin"], k, generator=g) / math.sqrt(s["Cin"] * k)
        b = torch.randn(s["Cout"], generator=g).to(DEV)
        fmt = pack.FMT_F16X2 if args.fmt == "f16x2" else pack.FMT_BF16X3
        nm = 3 if fmt == pack.FMT_F16X2 else 6
        wp, wt = pack.pack_conv(w.to(DEV)), pack.pack_conv_tc_planes(w.to(DEV), fmt)
        out = torch.empty(s["B"], s["T"], s["Cout"], device=DEV)
        flops = 2.0 * s["B"] * s["T"] * s["Cin"] * s["Cout"] * k
        ms = trace_ms(lambda: ops.conv1d(x, wp, b, out=out, w_tc=wt, k=k, dil=dil, pad=pad, pad_mode=1 if k > 1 else 0), reps)
        print(f"{s['name']:30s} {ms:8.3f} ms  {flops / ms / 1e9:7.1f} TFLOP/s fp32-equiv "
              f"({nm * flops / ms / 1e9:7.0f} dense 16-bit, {args.fmt})", flush=True)
        del x, out
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
