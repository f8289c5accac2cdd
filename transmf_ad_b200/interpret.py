"""Interpretability: Grad-CAM (Selvaraju et al., 2017) on a block of every sNet tower of a model, layer-wise relevance
propagation (Bach et al., 2015) and integrated gradients (Sundararajan et al., 2017) through the towers, and head-averaged
or gradient-weighted (Chefer et al., 2021) cross-modal attention maps of the fusion transformer.

Input gradients (saliency maps) need nothing from here: ``mri.requires_grad_(True)`` and plain autograd work on every model
(INTEGRATION.md section 3b).  Module hooks on the sNet blocks work as on the reference modules (section 3c), and so do
module hooks on ``Attention.attend`` (section 3d).
"""
from __future__ import annotations

from collections import namedtuple

import torch

from . import functional as TF
from .models.networks import BLOCKS, CrossTransformer, CrossTransformer_MOD_AVG, _has_backward_hooks, sNet


def _target_index(target, B, device, who="grad_cam"):
    if isinstance(target, int) and not isinstance(target, bool):
        return torch.full((B,), target, dtype=torch.long, device=device)
    if torch.is_tensor(target) and target.dim() <= 1 and not target.is_floating_point() and target.dtype != torch.bool:
        t = target.reshape(-1).to(device=device, dtype=torch.long)
        if t.numel() == 1:
            t = t.expand(B)
        if t.numel() == B:
            return t
    raise ValueError(f"{who}: target must be a class index or an integer tensor of shape ({B},); got {target!r}")


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


CrossAttention = namedtuple("CrossAttention", ["maps", "mri", "pet"])


def cross_attention(model, inputs, target=None, upsample=True, normalize=True):
    """Cross-modal attention maps of the fusion transformer of ``model`` (``CrossTransformer_MOD_AVG``: ``model_ad``,
    ``model_transformer``; ``CrossTransformer``: ``model_transformer_res``).

    Per encoder call, M[b,i,j] = mean_h attn (``target=None``: forward only) or mean_h max(attn * dL/d attn, 0) for the
    objective ``sum_b logits[b, target_b]`` of the model's first output (gradient-weighted, Chefer et al. 2021); a key
    token's relevance is r[b,j] = mean_i M[b,i,j].  Returns ``CrossAttention(maps, mri, pet)``:
      ``maps``: per layer, the (mri_enc, pet_enc) pair of fp32 (B, Nq, Nk) maps M;
      ``pet`` / ``mri``: fp32 (B,1,D,H,W) volume maps (``upsample``; else the tower output's (B,1,d,h,w)), normalised per
      sample to [0,1] (``normalize``).  ``CrossTransformer_MOD_AVG``: the PET map sums, over layers, the key relevance of
      ``mri_enc`` (where MRI queries looked in PET) and the MRI map that of ``pet_enc``.  ``CrossTransformer``: both
      encoders attend to cat([mri, pet]); the MRI map sums r[:, :N], the PET map r[:, N:], over layers and encoders.
    Key token n is the sNet output voxel (x, y, z) with n = (x*h + y)*w + z (``tokens_of``).

    The model runs in its current mode.  The towers run without autograd and their outputs become leaves, so no sNet
    backward runs; no parameter receives a ``.grad``, no weight-gradient kernel runs, and ``requires_grad`` flags are
    restored afterwards."""
    fusers = [m for m in model.modules() if isinstance(m, (CrossTransformer, CrossTransformer_MOD_AVG))]
    if not fusers:
        raise ValueError("cross_attention: the model has no fusion transformer (CrossTransformer or CrossTransformer_MOD_AVG)")
    if len(fusers) > 1:
        raise ValueError("cross_attention: the model has more than one fusion transformer")
    fuser = fusers[0]
    if isinstance(fuser, CrossTransformer) and fuser.share:
        raise ValueError("cross_attention: CrossTransformer(share=True) is not supported")
    towers = [m for m in model.modules() if isinstance(m, sNet)]
    inputs = tuple(inputs) if isinstance(inputs, (tuple, list)) else (inputs,)
    if len(inputs) != 2 or not all(torch.is_tensor(x) and x.dim() == 5 for x in inputs):
        raise ValueError("cross_attention: inputs must be the (mri, pet) pair of (B,1,D,H,W) volumes")
    B = inputs[0].shape[0]
    encs = [enc for pair in fuser.layers for enc in pair]              # reference order: mri_enc, pet_enc per layer
    probs, grid = {}, {}
    weighted = target is not None

    def keep_attn(i):
        def hook(module, args, attn):
            probs.setdefault(i, attn)
        return hook

    def leaf(module, args, out):
        grid["dhw"] = tuple(out.shape[2:])
        return out.detach().requires_grad_(True) if weighted else None

    flags = [(p, p.requires_grad) for p in model.parameters()]
    handles = []
    try:
        for p, _ in flags:
            p.requires_grad_(False)
        for i, enc in enumerate(encs):
            handles.append(enc.layers[0][0].fn.attend.register_forward_hook(keep_attn(i)))
        for t in towers:
            handles.append(t.register_forward_hook(leaf))
        with torch.enable_grad() if weighted else torch.no_grad():
            outs = model(*inputs)
            if len(probs) != len(encs) or "dhw" not in grid:
                raise RuntimeError("cross_attention: the fusion transformer or a tower did not run in the model's forward pass")
            attns = [probs[i] for i in range(len(encs))]
            grads = [None] * len(encs)
            if weighted:
                logits = outs[0] if isinstance(outs, (tuple, list)) else outs
                idx = _target_index(target, B, logits.device, "cross_attention")
                objective = logits.gather(1, idx.view(-1, 1)).sum()
                grads = list(torch.autograd.grad(objective, attns))
    finally:
        for h in handles:
            h.remove()
        for p, f in flags:
            p.requires_grad_(f)
    d, h, w = grid["dhw"]
    N = d * h * w
    maps = []
    if isinstance(fuser, CrossTransformer_MOD_AVG):
        r = torch.empty((2, B, N), dtype=torch.float32, device=attns[0].device)     # [mri map, pet map]
        for i, (a, g) in enumerate(zip(attns, grads)):
            # mri_enc (even i): MRI queries, PET keys -> the PET map; pet_enc: the MRI map
            M, _ = TF.attn_relevance(a, g, r[1 - i % 2], accumulate=i >= 2)
            maps.append(M)
        r = r.view(2, B, d, h, w)
    else:
        rr = torch.empty((B, 2 * N), dtype=torch.float32, device=attns[0].device)
        for i, (a, g) in enumerate(zip(attns, grads)):
            M, _ = TF.attn_relevance(a, g, rr, accumulate=i > 0)
            maps.append(M)
        r = torch.stack([rr[:, :N], rr[:, N:]]).view(2, B, d, h, w)
    size = tuple(inputs[0].shape[2:]) if upsample else (d, h, w)
    mri, pet = TF.map_resample(r, size, normalize)
    pairs = [(maps[2 * l], maps[2 * l + 1]) for l in range(len(maps) // 2)]
    return CrossAttention(pairs, mri, pet)


LRP = namedtuple("LRP", ["maps", "totals"])


def lrp(model, inputs, target, rule="epsilon", eps=1e-6, normalize=False):
    """Layer-wise relevance propagation (Bach et al., 2015) through every sNet tower of ``model`` (eval mode), for the
    objective f = ``sum_b logits[b, target_b]`` of the model's first output.

    The relevance at a tower output a_T is R_T = a_T * df/da_T (gradient x input: LRP-0 through the piecewise-linear heads);
    it is propagated through the seven conv units with BatchNorm folded into the convolutions (running statistics) and one
    ``rule`` for all of them: ``"epsilon"`` (LRP-eps; ``eps=0`` is LRP-0: the denominator is the pre-activation, bias
    included, stabilised as z + eps*sign(z)) or ``"zplus"`` (z+: the positive part of the folded weight, no bias).  LeakyReLU
    passes relevance unchanged, max-pool sends it to the first maximum of each window, the final avg-pool splits it in
    proportion to the activations.  ``inputs`` and ``target`` as for ``grad_cam``.

    Returns ``LRP(maps, totals)``: per tower, in tower order (``model.modules()``), an fp32 (B,1,D,H,W) signed relevance map
    (divided per sample by its max |R| with ``normalize``) and an fp32 (B, 8) tensor of per-sample relevance sums: at the
    tower output (column 0), then entering layers 6 .. 0 (columns 1 .. 7; column 7 is the sum of the map before
    normalisation).

    The towers run once, without autograd; no sNet backward runs, no parameter receives a ``.grad``, no weight-gradient
    kernel runs, BatchNorm buffers and the module mode are untouched and ``requires_grad`` flags are restored."""
    if rule not in TF.LRP_RULES:
        raise ValueError(f"lrp: rule must be one of {tuple(TF.LRP_RULES)}; got {rule!r}")
    if isinstance(eps, bool) or not isinstance(eps, (int, float)) or not eps >= 0 or eps == float("inf"):
        raise ValueError(f"lrp: eps must be a finite number >= 0; got {eps!r}")
    towers = [m for m in model.modules() if isinstance(m, sNet)]
    if not towers:
        raise ValueError("lrp: the model has no sNet tower")
    if any(m.training for m in towers):
        raise ValueError("lrp: BatchNorm is folded with its running statistics; call model.eval() first")
    inputs = tuple(inputs) if isinstance(inputs, (tuple, list)) else (inputs,)
    if not inputs or not all(torch.is_tensor(x) and x.dim() == 5 and x.shape[1] == 1 for x in inputs):
        raise ValueError("lrp: inputs must be (B,1,D,H,W) volumes")
    B = inputs[0].shape[0]
    idx = _target_index(target, B, inputs[0].device, "lrp")
    leaves = {}

    def leaf(module, args, out):
        o = out.detach().requires_grad_(True)
        leaves[module] = o
        return o

    flags = [(p, p.requires_grad) for p in model.parameters()]
    handles = []
    try:
        for p, _ in flags:
            p.requires_grad_(False)
        for t in towers:
            t._lrp_keep = []
            handles.append(t.register_forward_hook(leaf))
        with torch.enable_grad():
            outs = model(*[x.detach() for x in inputs])
            logits = outs[0] if isinstance(outs, (tuple, list)) else outs
            objective = logits.gather(1, idx.to(logits.device).view(-1, 1)).sum()
            acts = [leaves.get(t) for t in towers]
            kept = [t._lrp_keep for t in towers]
            if any(a is None for a in acts):
                raise RuntimeError("lrp: a tower of the model did not run in its forward pass")
            if any(len(k) != len(t._spec.layers) for k, t in zip(kept, towers)):
                raise RuntimeError("lrp: the towers did not run the folded eval path (TMF_EVAL_FOLD=0?)")
            grads = torch.autograd.grad(objective, acts, allow_unused=True)
    finally:
        for h in handles:
            h.remove()
        for p, f in flags:
            p.requires_grad_(f)
        for t in towers:
            t._lrp_keep = None
    seeds = [(TF._f32c(a.detach().permute(0, 2, 3, 4, 1)),
              TF._f32c(torch.zeros_like(a) if g is None else g.permute(0, 2, 3, 4, 1))) for a, g in zip(acts, grads)]
    maps, totals = [None] * len(towers), [None] * len(towers)
    i = 0
    while i < len(towers):
        grp = [i]
        if (i + 1 < len(towers) and towers[i + 1]._spec.dim == towers[i]._spec.dim
                and kept[i + 1][0][0].shape == kept[i][0][0].shape and towers[i + 1]._hyper() == towers[i]._hyper()):
            grp.append(i + 1)
        folds = [towers[t]._lrp_folds.setdefault(rule, [TF.LrpFold() for _ in range(7)]) for t in grp]
        params = []
        for t in grp:
            params.append([(conv.weight.detach(), conv.bias.detach(), bn.weight.detach(), bn.bias.detach(), bn.running_mean,
                            bn.running_var) for conv, bn in towers[t]._units()])
        m, tot = TF.lrp_towers(towers[i]._spec, towers[i]._hyper(), folds, params, [kept[t] for t in grp],
                               [seeds[t] for t in grp], rule, eps)
        for t, mm, tt in zip(grp, m, tot):
            maps[t], totals[t] = mm, tt
        i += len(grp)
    if normalize:
        TF.lrp_normalize(maps)
    return LRP(maps, totals)


IG = namedtuple("IG", ["maps", "delta"])
IG_METHODS = ("gausslegendre", "riemann_middle")


def ig_path(n_steps, method="gausslegendre"):
    """Path points and weights (alpha, w) of integrated gradients on [0, 1], float64 numpy arrays of ``n_steps``, as captum
    places them: ``"gausslegendre"`` maps numpy's ``leggauss`` nodes t to alpha = (1 + t) / 2 with w = w_t / 2;
    ``"riemann_middle"`` has alpha = (k + 1/2) / n and w = 1 / n.  Both put every alpha in (0, 1) and sum w to 1."""
    import numpy as np
    if method == "gausslegendre":
        t, wt = np.polynomial.legendre.leggauss(n_steps)
        return (1.0 + t) / 2.0, wt / 2.0
    k = np.arange(n_steps, dtype=np.float64)
    return (k + 0.5) / n_steps, np.full(n_steps, 1.0 / n_steps)


def _is_count(v):
    return isinstance(v, int) and not isinstance(v, bool) and v >= 1


def integrated_gradients(model, inputs, target, n_steps=50, method="gausslegendre", internal_batch_size=None):
    """Integrated gradients (Sundararajan et al., 2017) through every sNet tower of ``model`` (eval mode) with the zero
    baseline, for the objective f = ``logits[b, target_b]`` of the model's first output: IG = x * sum_k w_k df/dx(alpha_k x),
    with the path points of ``method`` (``ig_path``: ``"gausslegendre"``, captum's default, or ``"riemann_middle"``).
    ``inputs`` and ``target`` as for ``grad_cam``; tower t takes ``inputs[t]``.  ``internal_batch_size`` counts volumes per
    pass as captum does: max(1, internal_batch_size // B) path points go through the model together (``None``: all).

    Returns ``IG(maps, delta)``: per tower, in tower order (``model.modules()``), an fp32 (B,1,D,H,W) attribution map, and
    the fp32 (B,) convergence delta sum_towers sum_voxels maps - (f(x) - f(0)), with f(x) and f(0) from two eval forwards.

    Block 1 is factored out of the path integral (DESIGN section 3.10): for alpha > 0 its output at alpha x is
    LeakyReLU(alpha * umax + b') with the max-pool winners of u' = W' * x fixed, so conv1.0 runs once, the path points
    start at layer 1, and the block-1 input gradient runs once on the weighted sum of the path's gradients.  That is exact
    only for the zero baseline and alpha > 0: methods with a point at alpha = 0 (left / trapezoid Riemann sums) are
    refused, and so are non-zero baselines -- their winners move with alpha.  For those, captum's ``IntegratedGradients``
    works on these modules through plain autograd (INTEGRATION.md section 3b).

    No parameter receives a ``.grad``, no weight-gradient kernel runs, BatchNorm buffers and the module mode are untouched
    and ``requires_grad`` flags are restored."""
    who = "integrated_gradients"
    if method not in IG_METHODS:
        raise ValueError(f"{who}: method must be one of {IG_METHODS}; got {method!r} (left / trapezoid Riemann sums put a "
                         f"path point at alpha = 0, where every pooling window ties and block 1 cannot be factored out)")
    if not _is_count(n_steps):
        raise ValueError(f"{who}: n_steps must be an integer >= 1; got {n_steps!r}")
    if internal_batch_size is not None and not _is_count(internal_batch_size):
        raise ValueError(f"{who}: internal_batch_size must be None or an integer >= 1; got {internal_batch_size!r}")
    towers = [m for m in model.modules() if isinstance(m, sNet)]
    if not towers:
        raise ValueError(f"{who}: the model has no sNet tower")
    if any(m.training for m in model.modules()):
        raise ValueError(f"{who}: BatchNorm is folded with its running statistics; call model.eval() first")
    inputs = tuple(inputs) if isinstance(inputs, (tuple, list)) else (inputs,)
    if (len(inputs) != len(towers) or not all(torch.is_tensor(x) and x.dim() == 5 and x.shape[1] == 1 for x in inputs)
            or any(x.shape != inputs[0].shape for x in inputs)):
        raise ValueError(f"{who}: inputs must be {len(towers)} (B,1,D,H,W) volume(s) of one shape, one per tower")
    for t in towers:
        if t._forward_hooks or t._forward_pre_hooks or _has_backward_hooks(t) or t.conv1._forward_hooks \
                or t.conv1._forward_pre_hooks:
            raise ValueError(f"{who}: hooks on an sNet tower or its conv1 block would observe volumes that are never formed "
                             f"(the path points start at layer 1); remove them")
        if t._hyper()[0][2] < 0:
            raise ValueError(f"{who}: block 1's LeakyReLU slope must be >= 0 (the pooling winners must not move with alpha)")
    B = inputs[0].shape[0]
    idx = _target_index(target, B, inputs[0].device, who)
    if not all(x.is_cuda for x in inputs):
        raise ValueError(f"{who}: inputs must be CUDA tensors")
    alpha64, w64 = ig_path(n_steps, method)
    dev = inputs[0].device
    alpha = torch.tensor(alpha64, dtype=torch.float32, device=dev)
    weight = torch.tensor(w64, dtype=torch.float32, device=dev)
    chunk = n_steps if internal_batch_size is None else max(1, internal_batch_size // B)
    xs = [TF._f32c(x.detach()) for x in inputs]

    def objective(outs, rows):
        logits = outs[0] if isinstance(outs, (tuple, list)) else outs
        return logits.gather(1, rows.view(-1, 1)).view(-1)

    with torch.no_grad():
        f_x = objective(model(*xs), idx)
        f_0 = objective(model(*[torch.zeros_like(x) for x in xs]), idx)
    groups, i = [], 0
    while i < len(towers):
        grp = [i]
        if i + 1 < len(towers) and towers[i + 1]._spec.dim == towers[i]._spec.dim and towers[i + 1]._hyper() == towers[i]._hyper():
            grp.append(i + 1)
        groups.append(grp)
        i += len(grp)
    state = []
    for grp in groups:
        folds = [towers[t]._folds[0] for t in grp]
        units = [towers[t]._units()[0] for t in grp]
        tensors = [(c.weight, c.bias, bn.weight, bn.bias, bn.running_mean, bn.running_var) for c, bn in units]
        u, umax = TF.ig_block1([xs[t] for t in grp], folds, tensors, towers[grp[0]]._hyper()[0][0])
        G = [torch.zeros(m.shape, dtype=torch.float32, device=dev) for m in umax]
        state.append((folds, [f.bias for f in folds], u, umax, G, towers[grp[0]]._hyper()[0][2]))
    flags = [(p, p.requires_grad) for p in model.parameters()]
    try:
        for p, _ in flags:
            p.requires_grad_(False)
        for k0 in range(0, n_steps, chunk):
            m = min(chunk, n_steps - k0)
            a_k, w_k = alpha[k0:k0 + m], weight[k0:k0 + m]
            leaves = [None] * len(towers)
            for grp, (_, bias, _, umax, _, slope) in zip(groups, state):
                a16, a32 = TF.ig_expand(umax, bias, a_k, slope)
                for t, h, v in zip(grp, a16, a32):
                    leaves[t] = v.permute(0, 4, 1, 2, 3).detach().requires_grad_(True)
                    towers[t]._ig_src = (leaves[t], h)
            # zero-stride stand-ins of batch m*B: the towers start from the supplied block-1 outputs and never read them
            stand_ins = [x.as_strided((m * B,) + tuple(x.shape[1:]), (0,) * 5) for x in xs]
            with torch.enable_grad():
                obj = objective(model(*stand_ins), idx.repeat(m)).sum()
                grads = torch.autograd.grad(obj, leaves, allow_unused=True)
            for grp, (_, bias, _, umax, G, slope) in zip(groups, state):
                g = [TF._f32c((torch.zeros_like(leaves[t]) if grads[t] is None else grads[t]).permute(0, 2, 3, 4, 1))
                     for t in grp]
                TF.ig_combine(g, umax, bias, a_k, w_k, G, slope)
    finally:
        for p, f in flags:
            p.requires_grad_(f)
        for t in towers:
            t._ig_src = None
    maps, total = [None] * len(towers), torch.zeros_like(f_x)
    for grp, (folds, _, u, _, G, _) in zip(groups, state):
        dx = TF.ig_input_grad(G, u, folds)
        for t, m, s in zip(grp, dx, TF.ig_attribute([xs[t] for t in grp], dx)):
            maps[t] = m
            total = total + s
    return IG(maps, total - (f_x - f_0))
