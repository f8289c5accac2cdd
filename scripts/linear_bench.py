#!/usr/bin/env python
"""Linear-layer microbenchmark (B200): tmf_linear_fwd / dgrad / wgrad at the fusion transformer's shapes (M = B*150
tokens), CUDA events over `--iters` launches.  Every shape here runs gemm_ksplit_kernel; the generic gemm_kernel only
takes shapes with an extent that is not a multiple of 4.

    python scripts/linear_bench.py [--iters 50] [--batch 8]
"""
import argparse
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from transmf_ad_b200 import _lib as L          # noqa: E402

SHAPES = [("to_q/to_out", 128, 128), ("to_kv", 128, 256), ("ff1", 128, 512), ("ff2", 512, 128)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--batch", type=int, default=8)
    args = ap.parse_args()
    dev = "cuda"
    M = args.batch * 150
    tot = 0.0
    for name, K, N in SHAPES + [("head(M=B)", 512, 128)]:
        m = args.batch if name.startswith("head") else M
        x = torch.randn(m, K, device=dev)
        w = torch.randn(N, K, device=dev) * K ** -0.5
        b = torch.randn(N, device=dev)
        y, dy = torch.empty(m, N, device=dev), torch.randn(m, N, device=dev)
        dx, dw, db = torch.empty(m, K, device=dev), torch.empty(N, K, device=dev), torch.empty(N, device=dev)
        ops = {
            "fwd": lambda: L.call("tmf_linear_fwd", L.ptr(x), L.ptr(w), L.ptr(b), L.ptr(None), L.ptr(y), L.ptr(None), m, K, N, 0),
            "dgrad": lambda: L.call("tmf_linear_dgrad", L.ptr(dy), L.ptr(w), L.ptr(dx), m, K, N, 0),
            "wgrad": lambda: L.call("tmf_linear_wgrad", L.ptr(dy), L.ptr(x), L.ptr(dw), L.ptr(db), m, K, N, L.ptr(L.scratch("cuda")[0]), L.scratch("cuda")[1]),
        }
        for op, fn in ops.items():
            for _ in range(3):
                fn()
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()          # graph replay: device time without the Python launch cost
            with torch.cuda.graph(g):
                for _ in range(args.iters):
                    fn()
            g.replay()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            g.replay()
            e1.record()
            torch.cuda.synchronize()
            us = e0.elapsed_time(e1) / args.iters * 1e3
            tot += us if not name.startswith("head") else 0.0
            print(f"{name:12s} {op:5s} M={m:5d} K={K:4d} N={N:4d}: {us:7.2f} us  {2.0 * m * K * N / us / 1e6:6.2f} TFLOP/s", flush=True)
    print(f"sum over the transformer shapes: {tot:.1f} us (x6 encoders, to_q and to_out both once)")


if __name__ == "__main__":
    main()
