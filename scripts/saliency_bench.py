"""Input-gradient (saliency) measurements on one GPU, in one process:

  1. the block-1 input-gradient kernel alone (tmf_conv1_dgrad_fused, default impl) at B = 8 x 2 towers, 91 x 109 x 91:
     CUDA-event time, algorithmic bytes (y + pooled gradient read, dx written once) over that time, and its share of the
     6.45 TB/s device-to-device copy rate measured on B200 (DESIGN.md section 8);
  2. eval-mode saliency of model_ad with frozen weights: forward + backward to both volumes, subjects/s;
  3. the eager train step of model_ad with and without the volumes requiring grad (the cost of also asking for them);
  4. the GPU name and power limit, read in the same run (nvidia-smi query only).

Usage: python scripts/saliency_bench.py [--batch 8] [--iters 50] [--out FILE]   (prints one JSON object)
Inputs are far larger than the 126 MB L2 (y alone is 924 MB at B = 8), so every timed pass reads HBM.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from transmf_ad_b200 import _lib as L                                   # noqa: E402
from transmf_ad_b200.models import mymodel as M                        # noqa: E402
from transmf_ad_b200.synthetic import make_labels, make_volumes, procedural_state   # noqa: E402

SHAPE = (91, 109, 91)
COPY_PEAK = 6.45e12            # B/s, device-to-device copy, DESIGN.md section 8


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=60).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else "unavailable"
    except (OSError, subprocess.SubprocessError):
        return "unavailable"


def timed(fn, iters, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def kernel_alone(B, iters):
    D, H, W = SHAPE
    C, ng = 32, 2
    g = torch.Generator(device="cuda").manual_seed(0)
    ys = [torch.randn((B, D, H, W, C), device="cuda", generator=g).bfloat16() for _ in range(ng)]
    douts = [torch.randn((B, D // 2, H // 2, W // 2, C), device="cuda", generator=g).bfloat16() for _ in range(ng)]
    coefs = [torch.cat([torch.rand(C, device="cuda") + 0.5, torch.randn(C, device="cuda") * 0.1,
                        torch.randn(C, device="cuda") * 0.1, torch.rand(C, device="cuda") + 0.5]) for _ in range(ng)]
    bcoefs = [torch.randn(2 * C, device="cuda") * 0.01 for _ in range(ng)]
    ws = [torch.randn((C, 1, 3, 3, 3), device="cuda") * 0.2 for _ in range(ng)]
    dx = [torch.empty((B, D, H, W), device="cuda") for _ in range(ng)]
    impl = L.CONV_AUTO
    nws = int(L.load().tmf_conv1_dgrad_fused_workspace_bytes(ng, impl, B, D, H, W, C))
    buf = torch.empty(nws, dtype=torch.uint8, device="cuda") if nws > 0 else None
    args = (ng, L.ptrs(douts), L.ptrs(ys), L.ptrs(coefs), L.ptrs(bcoefs), L.ptrs(ws), L.ptrs(dx), B, D, H, W, C, 0.01, impl,
            L.ptr(buf), nws)
    ms = timed(lambda: L.call("tmf_conv1_dgrad_fused", *args), iters)
    vox = ng * B * D * H * W
    nbytes = vox * C * 2 + ng * B * (D // 2) * (H // 2) * (W // 2) * C * 2 + vox * 4
    return {"ms": round(ms, 4), "algorithmic_bytes": nbytes, "GB_per_s": round(nbytes / ms / 1e6, 1),
            "fraction_of_copy_peak": round(nbytes / (ms * 1e-3) / COPY_PEAK, 3), "workspace_bytes": nws}


def model_ad(B):
    model = M.model_ad(dim=128, depth=3, heads=4, dim_head=32, mlp_dim=512, dropout=0.0)
    model.load_state_dict(procedural_state(model.state_dict(), seed=0))
    label = make_labels(B)
    mri = make_volumes(B, SHAPE, seed=1, labels=label).cuda()
    pet = make_volumes(B, SHAPE, seed=2, labels=label).cuda()
    return model.cuda(), mri, pet, label.cuda()


def saliency(B, iters):
    model, mri, pet, label = model_ad(B)
    model.eval().requires_grad_(False)

    def step():
        a, b = mri.detach().requires_grad_(True), pet.detach().requires_grad_(True)
        logits = model(a, b)[0]
        torch.autograd.grad(logits.gather(1, label.view(-1, 1)).sum(), [a, b])

    ms = timed(step, iters)
    return {"ms_per_batch": round(ms, 3), "subjects_per_s": round(B / ms * 1e3, 1)}


def train_delta(B, iters):
    model, mri, pet, label = model_ad(B)
    model.train()
    opt = torch.optim.SGD(model.parameters(), lr=0.0)
    ce = torch.nn.CrossEntropyLoss()

    def step(want):
        a, b = mri.detach().requires_grad_(want), pet.detach().requires_grad_(want)
        logits, dm, dp = model(a, b)
        loss = ce(logits, label) + ce(dm, torch.zeros_like(label)) + ce(dp, torch.ones_like(label))
        opt.zero_grad(set_to_none=True)
        loss.backward()

    out = {}
    for rep in range(2):                       # alternate the two variants: drift of the shared host hits both
        for want in (False, True):
            ms = timed(lambda: step(want), iters)
            out.setdefault("with_input_grad" if want else "without", []).append(round(ms, 3))
    out["delta_ms"] = round(min(out["with_input_grad"]) - min(out["without"]), 3)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("saliency_bench.py measures on the GPU; no CUDA device found")
    res = {"gpu": gpu_info(), "torch_device": torch.cuda.get_device_name(), "batch": a.batch, "shape": SHAPE,
           "kernel_block1_input_grad_2towers": kernel_alone(a.batch, a.iters),
           "eval_saliency_model_ad_frozen": saliency(a.batch, max(5, a.iters // 5)),
           "train_step_model_ad_eager": train_delta(a.batch, max(5, a.iters // 5))}
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
