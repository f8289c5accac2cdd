"""Attention-map measurements on one GPU, in one process (DESIGN.md section 3.8):

  1. tmf_attn_scores in both modes next to tmf_attn_fwd, at B = 8, heads 4, dim_head 32 and (Nq, Nk) = (150, 150)
     (model_ad's encoders) and (150, 300) (model_transformer_res's): CUDA-event time per call over many calls;
  2. tmf_attn_relevance (gradient-weighted) + tmf_map_resample of two maps to 91 x 109 x 91 with normalisation;
  3. cross_attention(model_ad) in eval mode, subjects/s, without and with a target;
  4. the eager train step of model_ad with observing hooks (and tensor hooks on attn) on all six attend modules against
     the same step without hooks, alternated;
  5. the GPU name and power limit, read in the same run (nvidia-smi query only).

Usage: python scripts/attention_maps_bench.py [--batch 8] [--iters 200] [--out FILE]   (prints one JSON object)
The operands of 1 and 2 are a few MB and stay in the 126 MB L2: those kernel times are L2-resident figures.
"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from scripts.saliency_bench import SHAPE, gpu_info, model_ad, timed                # noqa: E402
from transmf_ad_b200 import _lib as L                                              # noqa: E402
from transmf_ad_b200 import functional as TF                                       # noqa: E402
from transmf_ad_b200.interpret import cross_attention                              # noqa: E402


def kernels(B, iters, heads=4, dh=32):
    g = torch.Generator(device="cuda").manual_seed(0)
    inner = heads * dh
    out = {}
    for Nq, Nk in ((150, 150), (150, 300)):
        q = torch.randn((B, Nq, inner), device="cuda", generator=g)
        kv = torch.randn((B, Nk, 2 * inner), device="cuda", generator=g)
        dout = torch.randn((B, Nq, inner), device="cuda", generator=g)
        o, lse = torch.empty_like(q), torch.empty((B, heads, Nq), device="cuda")
        dots, attn = torch.empty((2, B, heads, Nq, Nk), device="cuda").unbind(0)
        fwd = lambda: L.call("tmf_attn_fwd", L.ptr(q), L.ptr(kv), L.ptr(o), L.ptr(lse), B, Nq, Nk, heads, dh, dh ** -0.5)
        probs = lambda: L.call("tmf_attn_scores", 0, L.ptr(q), L.ptr(kv), L.ptr(lse), L.ptr(dots), L.ptr(attn), B, Nq, Nk,
                               heads, dh, dh ** -0.5)
        grad = lambda: L.call("tmf_attn_scores", 1, L.ptr(dout), L.ptr(kv), L.ptr(None), L.ptr(dots), L.ptr(None), B, Nq, Nk,
                              heads, dh, 1.0)
        fwd()
        rec = {}
        for name, fn in (("tmf_attn_fwd", fwd), ("scores_probs", probs), ("scores_grad", grad)):
            rec[name + "_us"] = round(timed(fn, iters) * 1e3, 2)
        nmap = B * heads * Nq * Nk * 4
        rec["probs_bytes_written"] = 2 * nmap
        rec["probs_GB_per_s"] = round(2 * nmap / (rec["scores_probs_us"] * 1e-6) / 1e9, 1)
        out[f"{Nq}x{Nk}"] = rec
    # relevance (gradient-weighted) of one encoder call + resampling of the two volume maps
    attn = torch.softmax(torch.randn((B, heads, 150, 150), device="cuda", generator=g), -1)
    dattn = torch.randn_like(attn)
    r = torch.empty((2, B, 150), device="cuda")
    rel = lambda: TF.attn_relevance(attn, dattn, r[0])
    res = lambda: TF.map_resample(r.view(2, B, 5, 6, 5), SHAPE, True)
    out["relevance_weighted_150x150_us"] = round(timed(rel, iters) * 1e3, 2)
    out["map_resample_2maps_normalized_us"] = round(timed(res, iters) * 1e3, 2)
    return out


def maps_throughput(B, iters):
    model, mri, pet, label = model_ad(B)
    model.eval()
    out = {}
    for name, target in (("plain", None), ("gradient_weighted", label)):
        ms = timed(lambda: cross_attention(model, (mri, pet), target), iters)
        out[name] = {"ms_per_batch": round(ms, 3), "subjects_per_s": round(B / ms * 1e3, 1)}
    return out


def train_hooks(B, iters):
    model, mri, pet, label = model_ad(B)
    model.train()
    opt = torch.optim.SGD(model.parameters(), lr=0.0)
    ce = torch.nn.CrossEntropyLoss()
    seen = []

    def hook(m, args, attn):
        seen.append(attn.shape)
        if attn.requires_grad:
            attn.register_hook(lambda g: seen.append(g.shape))

    def step():
        logits, dm, dp = model(mri, pet)
        loss = ce(logits, label) + ce(dm, torch.zeros_like(label)) + ce(dp, torch.ones_like(label))
        opt.zero_grad(set_to_none=True)
        loss.backward()
        seen.clear()

    attends = [enc.layers[0][0].fn.attend for pair in model.fuse_transformer.layers for enc in pair]
    out = {}
    for rep in range(3):                       # alternate the two variants: drift of the shared host hits both
        for hooked in (False, True):
            handles = [a.register_forward_hook(hook) for a in attends] if hooked else []
            ms = timed(step, iters)
            for hd in handles:
                hd.remove()
            out.setdefault("hooks_on_all_attend" if hooked else "without", []).append(round(ms, 3))
    out["delta_ms"] = round(min(out["hooks_on_all_attend"]) - min(out["without"]), 3)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("attention_maps_bench.py measures on the GPU; no CUDA device found")
    res = {"gpu": gpu_info(), "torch_device": torch.cuda.get_device_name(), "batch": a.batch, "shape": SHAPE,
           "kernels_b8_heads4_dh32": kernels(a.batch, a.iters),
           "cross_attention_model_ad_eval": maps_throughput(a.batch, max(5, a.iters // 20)),
           "train_step_model_ad_eager": train_hooks(a.batch, max(5, a.iters // 20))}
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
