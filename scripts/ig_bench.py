"""Integrated-gradients measurements on one GPU, in one process:

  1. interpret.integrated_gradients(model_ad) (block 1 factored out of the path integral) against a plain IG through the
     saliency path (the alpha_k x volumes batched through the model, autograd to the volumes), with the same chunking,
     alternated three times: ms per batch and subjects/s, and the relative L2 distance of the two maps;
  2. tmf_ig_expand / tmf_ig_combine for one chunk of both towers, by CUDA events, with their algorithmic bytes as a share of
     the 6.45 TB/s device-to-device copy rate measured on B200 (DESIGN.md section 8);
  3. the GPU name and power limit, read in the same run (nvidia-smi query only).

Usage: python scripts/ig_bench.py [--batch 8] [--steps 32] [--internal-batch 64] [--iters 20] [--out FILE]
Defaults: B = 8 subjects of 91 x 109 x 91, 32 Gauss-Legendre steps, 64 volumes per pass (8 path points per chunk).  Every
chunk moves gigabytes, far beyond the 126 MB L2, so the timed passes read HBM.
"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from saliency_bench import COPY_PEAK, SHAPE, gpu_info, model_ad, timed   # noqa: E402
from transmf_ad_b200 import functional as TF                             # noqa: E402
from transmf_ad_b200.interpret import ig_path, integrated_gradients      # noqa: E402


def plain_ig(model, xs, target, n, chunk):
    """IG through the saliency path, as a user builds it by hand."""
    alpha, w = ig_path(n)
    B = xs[0].shape[0]
    acc = [torch.zeros_like(x) for x in xs]
    for k0 in range(0, n, chunk):
        m = min(chunk, n - k0)
        a = torch.tensor(alpha[k0:k0 + m], dtype=torch.float32, device="cuda").view(-1, 1, 1, 1, 1, 1)
        wk = torch.tensor(w[k0:k0 + m], dtype=torch.float32, device="cuda").view(-1, 1, 1, 1, 1, 1)
        X = [(a * x.unsqueeze(0)).reshape((m * B,) + tuple(x.shape[1:])).requires_grad_(True) for x in xs]
        obj = model(*X)[0].gather(1, target.repeat(m).view(-1, 1)).sum()
        for t, g in enumerate(torch.autograd.grad(obj, X)):
            acc[t] += (wk * g.view((m,) + tuple(xs[t].shape))).sum(0)
    return [x * a for x, a in zip(xs, acc)]


def end_to_end(B, n, ibs):
    model, mri, pet, label = model_ad(B)
    model.eval().requires_grad_(False)
    xs = [mri, pet]
    chunk = max(1, ibs // B)
    fact = lambda: integrated_gradients(model, xs, label, n_steps=n, internal_batch_size=ibs)
    plain = lambda: plain_ig(model, xs, label, n, chunk)
    a, b = fact().maps, plain()
    rel = [float((x.double() - y.double()).norm() / y.double().norm()) for x, y in zip(a, b)]
    out = {"factored_ms": [], "plain_ms": []}
    for _ in range(3):                         # alternate: drift of the shared host hits both
        out["factored_ms"].append(round(timed(fact, 3, warmup=1), 2))
        out["plain_ms"].append(round(timed(plain, 3, warmup=1), 2))
    f, p = min(out["factored_ms"]), min(out["plain_ms"])
    out.update(factored_subjects_per_s=round(B / f * 1e3, 2), plain_subjects_per_s=round(B / p * 1e3, 2),
               speedup=round(p / f, 3), target_speedup=1.5, target_met=p / f >= 1.5,
               rel_l2_factored_vs_plain=[round(r, 5) for r in rel], points_per_chunk=chunk)
    return out


def kernels(B, chunk, iters):
    D, H, W = (s // 2 for s in SHAPE)
    C, ng = 32, 2
    g = torch.Generator(device="cuda").manual_seed(0)
    umax = [torch.randn((B, D, H, W, C), device="cuda", generator=g).bfloat16() for _ in range(ng)]
    bias = [torch.randn(C, device="cuda", generator=g) * 0.1 for _ in range(ng)]
    alpha = torch.rand(chunk, device="cuda", generator=g)
    w = torch.rand(chunk, device="cuda", generator=g)
    grads = [torch.randn((chunk * B, D, H, W, C), device="cuda", generator=g) for _ in range(ng)]
    G = [torch.zeros((B, D, H, W, C), device="cuda") for _ in range(ng)]
    el = ng * B * D * H * W * C
    exp_ms = timed(lambda: TF.ig_expand(umax, bias, alpha, 0.01), iters)
    comb_ms = timed(lambda: TF.ig_combine(grads, umax, bias, alpha, w, G, 0.01), iters)
    exp_bytes = el * 2 + chunk * el * (2 + 4)                 # umax once; a1 (bf16) and its fp32 twin per step
    comb_bytes = el * 2 + chunk * el * 4 + 2 * el * 4         # umax once, the chunk's gradients, G read and written

    def rec(ms, nbytes):
        return {"ms": round(ms, 4), "algorithmic_bytes": nbytes, "GB_per_s": round(nbytes / ms / 1e6, 1),
                "fraction_of_copy_peak": round(nbytes / (ms * 1e-3) / COPY_PEAK, 3)}

    return {"points_per_chunk": chunk, "towers": ng, "tmf_ig_expand": rec(exp_ms, exp_bytes),
            "tmf_ig_combine": rec(comb_ms, comb_bytes)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--steps", type=int, default=32)
    ap.add_argument("--internal-batch", type=int, default=64)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ig_bench.py measures on the GPU; no CUDA device found")
    res = {"gpu": gpu_info(), "torch_device": torch.cuda.get_device_name(), "batch": a.batch, "shape": SHAPE,
           "n_steps": a.steps, "method": "gausslegendre", "internal_batch_size": a.internal_batch,
           "model_ad_eval": end_to_end(a.batch, a.steps, a.internal_batch),
           "kernels": kernels(a.batch, max(1, a.internal_batch // a.batch), a.iters)}
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
