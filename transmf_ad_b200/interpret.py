"""Interpretability on the sNet towers: Grad-CAM (Selvaraju et al., 2017) on a block of every tower of a model.

Input gradients (saliency maps) need nothing from here: ``mri.requires_grad_(True)`` and plain autograd work on every model
(INTEGRATION.md section 3b).  Module hooks on the sNet blocks work as on the reference modules (section 3c).
"""
from __future__ import annotations

import torch

from . import functional as TF
from .models.networks import BLOCKS, sNet


def _target_index(target, B, device):
    if isinstance(target, int) and not isinstance(target, bool):
        return torch.full((B,), target, dtype=torch.long, device=device)
    if torch.is_tensor(target) and target.dim() <= 1 and not target.is_floating_point() and target.dtype != torch.bool:
        t = target.reshape(-1).to(device=device, dtype=torch.long)
        if t.numel() == 1:
            t = t.expand(B)
        if t.numel() == B:
            return t
    raise ValueError(f"grad_cam: target must be a class index or an integer tensor of shape ({B},); got {target!r}")


def grad_cam(model, inputs, target, layer="conv3", upsample=True, normalize=True):
    """Grad-CAM of ``layer`` (one of ``conv1`` ... ``conv4``) in every sNet tower of ``model``, for the objective
    ``sum_b logits[b, target_b]`` of the model's first output.

    ``inputs``: the volumes of ``model(*inputs)`` (a tensor for a one-tower model); ``target``: a class index or a (B,)
    integer tensor.  Returns one fp32 (B,1,D,H,W) map per tower, in tower order (``model.modules()``): upsampled to the
    input extent (``upsample``; else the block's extent) and normalised per sample to [0,1] (``normalize``).

    The model runs in its current mode.  The towers up to the block run without autograd, no parameter receives a
    ``.grad`` and no weight-gradient kernel runs; ``requires_grad`` flags are restored afterwards."""
    if layer not in BLOCKS:
        raise ValueError(f"grad_cam: layer must be one of {BLOCKS}; got {layer!r}")
    towers = [m for m in model.modules() if isinstance(m, sNet)]
    if not towers:
        raise ValueError("grad_cam: the model has no sNet tower")
    inputs = tuple(inputs) if isinstance(inputs, (tuple, list)) else (inputs,)
    if not inputs or not all(torch.is_tensor(x) and x.dim() == 5 for x in inputs):
        raise ValueError("grad_cam: inputs must be (B,1,D,H,W) volumes")
    B = inputs[0].shape[0]
    k = BLOCKS.index(layer)
    flags = [(p, p.requires_grad) for p in model.parameters()]
    try:
        for p, _ in flags:
            p.requires_grad_(False)
        for t in towers:
            t._cam_tap, t._cam_act = k, None
        with torch.enable_grad():
            outs = model(*inputs)
            logits = outs[0] if isinstance(outs, (tuple, list)) else outs
            idx = _target_index(target, B, logits.device)
            objective = logits.gather(1, idx.view(-1, 1)).sum()
            acts = [t._cam_act for t in towers]
            if any(a is None for a in acts):
                raise RuntimeError("grad_cam: a tower of the model did not run in its forward pass")
            grads = torch.autograd.grad(objective, acts)
    finally:
        for p, f in flags:
            p.requires_grad_(f)
        for t in towers:
            t._cam_tap, t._cam_act = None, None
    size = tuple(inputs[0].shape[2:]) if upsample else None
    return TF.gradcam(acts, grads, size=size, normalize=normalize)
