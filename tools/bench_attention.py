"""Attention time per shape (diagnostics, GPU only) at the PLM / ADM head shapes, sequence lengths 32 .. 512, through the
default dispatch: the fp32 kernel (ops.cu) up to 64 queries, the tcgen05 kernel (attn_tc.cu) above."""
import os
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from megatts2_b200 import ops  # noqa: E402


def main():
    for (B, H, dh) in ((64, 16, 64), (64, 8, 96), (16, 16, 64)):
        for S in [int(x) for x in os.environ.get("BENCH_S", "32,64,128,256,512").split(",")]:
            if B * S > 64 * 256 and B == 64:
                continue
            qkv = torch.randn(B, S, 3 * H * dh, device="cuda")
            D = H * dh
            f = lambda: ops.attention(qkv[..., :D], qkv[..., D:2 * D], qkv[..., 2 * D:], H)
            for _ in range(3):
                f()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(20):
                f()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / 20
            fl = 4.0 * B * H * S * S * dh
            print(f"B{B} H{H} dh{dh} S{S:4d}: {ms * 1e3:8.1f} us  {fl / ms / 1e9:7.2f} TFLOP/s", flush=True)


if __name__ == "__main__":
    main()
