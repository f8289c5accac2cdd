"""Grad-CAM measurements on one GPU, in one process:

  1. the Grad-CAM kernel alone (tmf_gradcam, upsampled to 91 x 109 x 91 and normalised) at B = 8 x 2 towers for each
     sNet block: CUDA-event time, algorithmic bytes (A and G read once, the map written once) over that time, and its
     share of the 6.45 TB/s device-to-device copy rate measured on B200 (DESIGN.md section 8);
  2. grad_cam(model_ad, layer) in eval mode with frozen weights, per block, subjects/s, next to eval saliency measured in
     the same run (scripts/saliency_bench.py; 1197 subjects/s in DESIGN.md section 3.4);
  3. the eager train step of model_ad with observing forward hooks on conv3 of both towers against the same step
     without hooks, alternated;
  4. the GPU name and power limit, read in the same run (nvidia-smi query only).

Usage: python scripts/gradcam_bench.py [--batch 8] [--iters 50] [--out FILE]   (prints one JSON object)
At conv1 A and G are 448 MB, far above the 126 MB L2; at conv3 / conv4 (3.5 / 0.4 MB) the kernel times are L2-resident
figures and say so in the record.
"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from scripts.saliency_bench import COPY_PEAK, SHAPE, gpu_info, model_ad, saliency, timed   # noqa: E402
from transmf_ad_b200 import functional as TF                                      # noqa: E402
from transmf_ad_b200.interpret import grad_cam                                    # noqa: E402
from transmf_ad_b200.models.networks import BLOCKS                                # noqa: E402

BLOCK_SHAPES = {"conv1": (32, 45, 54, 45), "conv2": (64, 22, 27, 22), "conv3": (128, 11, 13, 11), "conv4": (128, 5, 6, 5)}
L2_BYTES = 126 * 2 ** 20


def kernel_alone(B, iters):
    out = {}
    g = torch.Generator(device="cuda").manual_seed(0)
    for name in BLOCKS:
        C, d, h, w = BLOCK_SHAPES[name]
        mk = lambda: torch.randn((B, d, h, w, C), device="cuda", generator=g).permute(0, 4, 1, 2, 3)
        acts, grads = [mk().abs() for _ in range(2)], [mk() for _ in range(2)]
        ms = timed(lambda: TF.gradcam(acts, grads, size=SHAPE, normalize=True), iters)
        nin = 2 * 2 * B * d * h * w * C * 4
        nbytes = nin + 2 * B * SHAPE[0] * SHAPE[1] * SHAPE[2] * 4
        out[name] = {"ms": round(ms, 4), "algorithmic_bytes": nbytes, "GB_per_s": round(nbytes / ms / 1e6, 1),
                     "fraction_of_copy_peak": round(nbytes / (ms * 1e-3) / COPY_PEAK, 3),
                     "inputs_fit_l2": nin < L2_BYTES}
    return out


def eval_gradcam(B, iters):
    model, mri, pet, label = model_ad(B)
    model.eval().requires_grad_(False)
    out = {}
    for name in BLOCKS:
        ms = timed(lambda: grad_cam(model, (mri, pet), label, layer=name), iters)
        out[name] = {"ms_per_batch": round(ms, 3), "subjects_per_s": round(B / ms * 1e3, 1)}
    return out


def train_hooks(B, iters):
    model, mri, pet, label = model_ad(B)
    model.train()
    opt = torch.optim.SGD(model.parameters(), lr=0.0)
    ce = torch.nn.CrossEntropyLoss()
    seen = []

    def step():
        logits, dm, dp = model(mri, pet)
        loss = ce(logits, label) + ce(dm, torch.zeros_like(label)) + ce(dp, torch.ones_like(label))
        opt.zero_grad(set_to_none=True)
        loss.backward()
        seen.clear()

    out = {}
    for rep in range(2):                       # alternate the two variants: drift of the shared host hits both
        for hooked in (False, True):
            handles = [t.conv3.register_forward_hook(lambda m, i, o: seen.append(o.shape))
                       for t in (model.mri_cnn, model.pet_cnn)] if hooked else []
            ms = timed(step, iters)
            for hd in handles:
                hd.remove()
            out.setdefault("hooks_on_conv3" if hooked else "without", []).append(round(ms, 3))
    out["delta_ms"] = round(min(out["hooks_on_conv3"]) - min(out["without"]), 3)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("gradcam_bench.py measures on the GPU; no CUDA device found")
    res = {"gpu": gpu_info(), "torch_device": torch.cuda.get_device_name(), "batch": a.batch, "shape": SHAPE,
           "kernel_gradcam_2towers_upsampled_normalized": kernel_alone(a.batch, a.iters),
           "eval_gradcam_model_ad_frozen": eval_gradcam(a.batch, max(5, a.iters // 5)),
           "eval_saliency_model_ad_frozen": saliency(a.batch, max(5, a.iters // 5)),
           "train_step_model_ad_eager": train_hooks(a.batch, max(5, a.iters // 5))}
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
