"""Layer-wise relevance propagation measurements on one GPU, in one process:

  1. the block-1 relevance kernel (tmf_lrp_conv1, default impl, rule epsilon) against the block-1 input-gradient kernel
     (tmf_conv1_dgrad_fused) at B = 8 x 2 towers, 91 x 109 x 91, alternated in the same run: CUDA-event times and their ratio;
  2. lrp(model_ad) for the rules epsilon and zplus, subjects/s, next to frozen-weight eval saliency (forward + backward to
     both volumes) in the same run;
  3. the GPU name and power limit, read in the same run (nvidia-smi query only).

Usage: python scripts/lrp_bench.py [--batch 8] [--iters 50] [--out FILE]   (prints one JSON object)
Inputs are far larger than the 126 MB L2 (y alone is 924 MB at B = 8), so every timed pass reads HBM.
"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from saliency_bench import SHAPE, gpu_info, model_ad, saliency, timed   # noqa: E402
from transmf_ad_b200 import _lib as L                                   # noqa: E402
from transmf_ad_b200.interpret import lrp                               # noqa: E402


def kernels(B, iters):
    D, H, W = SHAPE
    C, ng = 32, 2
    g = torch.Generator(device="cuda").manual_seed(0)
    ys = [torch.randn((B, D, H, W, C), device="cuda", generator=g).bfloat16() for _ in range(ng)]
    pooled = lambda: [torch.randn((B, D // 2, H // 2, W // 2, C), device="cuda", generator=g).bfloat16() for _ in range(ng)]
    douts, a1 = pooled(), pooled()
    coefs = [torch.cat([torch.rand(C, device="cuda") + 0.5, torch.randn(C, device="cuda") * 0.1,
                        torch.randn(C, device="cuda") * 0.1, torch.rand(C, device="cuda") + 0.5]) for _ in range(ng)]
    bcoefs = [torch.randn(2 * C, device="cuda") * 0.01 for _ in range(ng)]
    ws = [torch.randn((C, 1, 3, 3, 3), device="cuda") * 0.2 for _ in range(ng)]
    xs = [torch.randn((B, D, H, W), device="cuda") for _ in range(ng)]
    out = [torch.empty((B, D, H, W), device="cuda") for _ in range(ng)]
    tot = [torch.empty((B, 8), device="cuda") for _ in range(ng)]
    impl = L.CONV_AUTO
    n1 = int(L.load().tmf_conv1_dgrad_fused_workspace_bytes(ng, impl, B, D, H, W, C))
    b1 = torch.empty(max(n1, 1), dtype=torch.uint8, device="cuda")
    n2 = int(L.load().tmf_lrp_conv1_workspace_bytes(ng, impl, B, D, H, W, C))
    b2 = torch.empty(max(n2, 1), dtype=torch.uint8, device="cuda")
    sal = (ng, L.ptrs(douts), L.ptrs(ys), L.ptrs(coefs), L.ptrs(bcoefs), L.ptrs(ws), L.ptrs(out), B, D, H, W, C, 0.01, impl,
           L.ptr(b1), n1)
    rel = (ng, L.ptrs(a1), L.ptrs(douts), L.ptrs(ys), L.ptrs(None), L.ptrs(ws), L.ptrs(xs), L.ptrs(out), L.ptrs(tot), B, D, H,
           W, C, 1e-6, impl, L.ptr(b2), n2)
    res = {"tmf_conv1_dgrad_fused_ms": [], "tmf_lrp_conv1_ms": []}
    for _ in range(3):                         # alternate: drift of the shared host hits both
        res["tmf_conv1_dgrad_fused_ms"].append(round(timed(lambda: L.call("tmf_conv1_dgrad_fused", *sal), iters), 4))
        res["tmf_lrp_conv1_ms"].append(round(timed(lambda: L.call("tmf_lrp_conv1", *rel), iters), 4))
    res["ratio"] = round(min(res["tmf_lrp_conv1_ms"]) / min(res["tmf_conv1_dgrad_fused_ms"]), 3)
    res["impl"] = int(L.load().tmf_lrp_conv1_impl(ng, impl, B, D, H, W, C))
    return res


def model_rates(B, iters):
    model, mri, pet, label = model_ad(B)
    model.eval()
    out = {}
    for rep in range(2):
        out.setdefault("saliency_subjects_per_s", []).append(saliency(B, iters)["subjects_per_s"])
        for rule in ("epsilon", "zplus"):
            ms = timed(lambda: lrp(model, (mri, pet), label, rule=rule), iters)
            out.setdefault(f"lrp_{rule}_subjects_per_s", []).append(round(B / ms * 1e3, 1))
    best = {k: max(v) for k, v in out.items()}
    out["epsilon_vs_saliency"] = round(best["lrp_epsilon_subjects_per_s"] / best["saliency_subjects_per_s"], 3)
    out["zplus_vs_saliency"] = round(best["lrp_zplus_subjects_per_s"] / best["saliency_subjects_per_s"], 3)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("lrp_bench.py needs a CUDA device")
    res = {"gpu": gpu_info(), "torch_device": torch.cuda.get_device_name(), "batch": args.batch, "shape": list(SHAPE),
           "block1_2towers": kernels(args.batch, args.iters), "model_ad_eval": model_rates(args.batch, max(args.iters // 5, 5))}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
