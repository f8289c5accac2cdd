"""Interpretability: Grad-CAM (Selvaraju et al., 2017) on a block of every sNet tower of a model, layer-wise relevance
propagation (Bach et al., 2015), integrated gradients (Sundararajan et al., 2017), occlusion sensitivity (Zeiler & Fergus,
2014), feature ablation and Shapley value sampling (Castro et al., 2009) over the regions of a mask through the towers, and
head-averaged or gradient-weighted (Chefer et al., 2021) cross-modal attention maps of the fusion transformer.

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
        if not t.conv1[2].negative_slope >= 0:          # before sNet._hyper, which refuses any negative slope
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


Occlusion = namedtuple("Occlusion", ["maps", "scores"])


def _refuse_tower_hooks(towers, who, what):
    for t in towers:
        for mod in [t] + [getattr(t, name) for name in BLOCKS]:
            if mod._forward_hooks or mod._forward_pre_hooks or _has_backward_hooks(mod):
                raise ValueError(f"{who}: hooks on an sNet tower or its blocks would observe tensors that are never formed "
                                 f"(the {what} towers run on crops); remove them")


def _tower_groups(towers):
    """Runs of at most two consecutive towers of one shape, which go through the crop launches as one group."""
    groups, i = [], 0
    while i < len(towers):
        grp = [i]
        if i + 1 < len(towers) and towers[i + 1]._spec.dim == towers[i]._spec.dim and towers[i + 1]._hyper() == towers[i]._hyper():
            grp.append(i + 1)
        groups.append(grp)
        i += len(grp)
    return groups


def _objective(outs, rows):
    logits = outs[0] if isinstance(outs, (tuple, list)) else outs
    return logits.gather(1, rows.view(-1, 1)).view(-1)


def _base_forward(model, towers, xs, idx, who):
    """The unchanged eval forward that incremental recomputation starts from: f(x), every tower's kept (input activation, y)
    pairs and its fp32 (B, d, h, w, C) output.  Sets ``_lrp_keep`` on the towers; the caller clears it."""
    outs = {}

    def keep_out(module, args, out):
        outs[module] = out

    handles = []
    try:
        for t in towers:
            t._lrp_keep = []
            handles.append(t.register_forward_hook(keep_out))
        with torch.no_grad():
            f_x = _objective(model(*xs), idx)
    finally:
        for h in handles:
            h.remove()
    kept = [t._lrp_keep for t in towers]
    if any(t not in outs for t in towers):
        raise RuntimeError(f"{who}: a tower of the model did not run in its forward pass")
    if any(len(k) != len(t._spec.layers) for k, t in zip(kept, towers)):
        raise RuntimeError(f"{who}: the towers did not run the folded eval path (TMF_EVAL_FOLD=0?)")
    return f_x, kept, [TF._f32c(outs[t].permute(0, 2, 3, 4, 1)) for t in towers]


def _through_fusion(model, towers, xs, base, bufs, tab_out, m, extent, idx, blocks):
    """The end of a pass whose tower outputs are composed into ``bufs`` (per tower, fp32 rows blocks*m*B): with blocks > 1,
    row block u changed tower u only, and the other towers' outputs there are replicated from their base outputs; then the
    model's own fusion stack and heads.  Returns the objective on the rows, (blocks, m, B)."""
    nt, B = len(towers), xs[0].shape[0]
    reps = [(t, u) for t in range(nt) for u in range(nt) if u != t] if blocks > 1 else []
    while reps:
        pair = reps[:2] if len(reps) > 1 and base[reps[0][0]].shape == base[reps[1][0]].shape else reps[:1]
        TF.occ_compose([base[t] for t, _ in pair], None, tab_out, m, extent,
                       out=[bufs[t][u * m * B:(u + 1) * m * B] for t, u in pair], tag="tmf_occ_compose@base")
        reps = reps[len(pair):]
    for t, buf in zip(towers, bufs):
        t._occ_out = buf.permute(0, 4, 1, 2, 3)
    # zero-stride stand-ins of batch rows: the towers return their composed outputs and never read them
    stand_ins = [x.as_strided((blocks * m * B,) + tuple(x.shape[1:]), (0,) * 5) for x in xs]
    with torch.no_grad():
        return _objective(model(*stand_ins), idx.repeat(blocks * m)).view(blocks, m, B)


def _triple(v, who, name):
    v = (v,) * 3 if isinstance(v, int) and not isinstance(v, bool) else v
    if not (isinstance(v, (tuple, list)) and len(v) == 3 and all(_is_count(e) for e in v)):
        raise ValueError(f"{who}: {name} must be an integer >= 1 or a 3-tuple of them; got {v!r}")
    return tuple(v)


def occlusion(model, inputs, target, window=16, stride=8, baseline=0.0, internal_batch_size=None):
    """Occlusion sensitivity (Zeiler & Fergus, 2014) through every sNet tower of ``model`` (eval mode), for the objective
    f = ``logits[b, target_b]`` of the model's first output.  A box of ``window`` voxels set to ``baseline`` (a finite Python
    scalar) slides over tower t's input ``inputs[t]`` with ``stride``, the other inputs unchanged; along an axis of extent E,
    window i covers [i*s, i*s + w) for i = 0 .. (E - w) // s, as captum's ``Occlusion`` places them.  ``window`` and ``stride``:
    an int or a 3-tuple.  ``inputs`` and ``target`` as for ``integrated_gradients``.  ``internal_batch_size`` counts volumes per
    pass: max(1, internal_batch_size // B) windows of every tower go through the model together (``None``: all of them, split
    only where a kernel's 32-bit index limit requires it).

    Returns ``Occlusion(maps, scores)``, per tower in tower order (``model.modules()``): ``scores`` fp32 (B, nD, nH, nW),
    f(x) - f(x with window (i, j, k) of that tower's input set to the baseline); ``maps`` fp32 (B,1,D,H,W), each voxel's mean
    score over the windows that contain it (0 where none does).

    The occluded towers are not run in full (DESIGN section 3.11): one eval forward keeps every layer's input activation,
    and per window only the region the window changes is recomputed, layer by layer, on fixed-extent crops batched over the
    windows; the composed tower outputs then go through the model's own fusion stack and heads.  No parameter receives a
    ``.grad``, no weight-gradient kernel runs, BatchNorm buffers and the module mode are untouched and ``requires_grad``
    flags are restored."""
    import math
    who = "occlusion"
    window, stride = _triple(window, who, "window"), _triple(stride, who, "stride")
    if isinstance(baseline, bool) or not isinstance(baseline, (int, float)) or not math.isfinite(baseline):
        raise ValueError(f"{who}: baseline must be a finite Python scalar; got {baseline!r}")
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
    _refuse_tower_hooks(towers, who, "occluded")
    B, dims = inputs[0].shape[0], tuple(inputs[0].shape[2:])
    if any(w > E for w, E in zip(window, dims)):
        raise ValueError(f"{who}: window {window} is larger than the volume {dims}")
    idx = _target_index(target, B, inputs[0].device, who)
    if not all(x.is_cuda for x in inputs):
        raise ValueError(f"{who}: inputs must be CUDA tensors")
    dev = inputs[0].device
    xs = [TF._f32c(x.detach()) for x in inputs]
    spec = towers[0]._spec
    plan = TF.OccPlan(dims, window, stride, [(ks, pool) for _, _, ks, pool in spec.layers])
    groups = _tower_groups(towers)
    nt, nwin = len(towers), plan.nwin
    chunk = nwin if internal_batch_size is None else max(1, internal_batch_size // B)
    chunk = min([chunk] + [TF.occ_pass_limit(plan, towers[g[0]]._spec, B, len(g)) for g in groups])

    flags = [(p, p.requires_grad) for p in model.parameters()]
    try:
        for p, _ in flags:
            p.requires_grad_(False)
        f_x, kept, base = _base_forward(model, towers, xs, idx, who)
        tabs = [torch.from_numpy(tb).to(dev) for tb in plan.tab]          # ordinary host-to-device copies
        scores = torch.empty((nt, nwin, B), dtype=torch.float32, device=dev)
        for n0 in range(0, nwin, chunk):
            m = min(chunk, nwin - n0)
            rows = nt * m * B
            # rows [u*m*B, (u+1)*m*B) occlude tower u's input: tower u's output there is composed, the others' replicated
            bufs = [torch.empty((rows,) + plan.crop[-1] + (b.shape[-1],), dtype=torch.float32, device=dev) for b in base]
            tab = [tb[n0:n0 + m] for tb in tabs]
            for grp in groups:
                TF.occ_towers(towers[grp[0]]._spec, towers[grp[0]]._hyper(), [towers[t]._folds for t in grp],
                              [xs[t] for t in grp], [kept[t] for t in grp], [base[t] for t in grp], plan, tab, m, baseline,
                              [bufs[t][t * m * B:(t + 1) * m * B] for t in grp])
            f_occ = _through_fusion(model, towers, xs, base, bufs, tab[-1], m, plan.crop[-1], idx, nt)
            scores[:, n0:n0 + m] = f_x.view(1, 1, B) - f_occ
    finally:
        for p, f in flags:
            p.requires_grad_(f)
        for t in towers:
            t._lrp_keep = None
            t._occ_out = None
    per = [s.t().reshape((B,) + plan.grid).contiguous() for s in scores.unbind(0)]
    return Occlusion(TF.occ_map(per, plan), per)


FeatureAblation = namedtuple("FeatureAblation", ["maps", "scores"])


def _ablation_baselines(baselines, nt, shape, device, who):
    """Per tower a float or an fp32 contiguous (1|B,1,D,H,W) tensor, from a scalar or a tuple of one entry per tower."""
    import math

    def scalar(b):
        return isinstance(b, (int, float)) and not isinstance(b, bool) and math.isfinite(b)

    if not isinstance(baselines, (tuple, list)):
        if not scalar(baselines):
            raise ValueError(f"{who}: baselines must be a finite Python scalar or a tuple of {nt} entries, one per tower; "
                             f"got {baselines!r}")
        return [float(baselines)] * nt
    if len(baselines) != nt:
        raise ValueError(f"{who}: baselines must be a scalar or a tuple of {nt} entries, one per tower; got {len(baselines)}")
    out = []
    for b in baselines:
        if scalar(b):
            out.append(float(b))
        elif (torch.is_tensor(b) and b.dtype == torch.float32 and b.device == device and b.dim() == 5
              and b.shape[0] in (1, shape[0]) and tuple(b.shape[1:]) == tuple(shape[1:])):
            out.append(b.detach().contiguous())
        else:
            raise ValueError(f"{who}: each baseline must be a finite Python scalar or an fp32 tensor of shape "
                             f"(1|{shape[0]}, 1, {', '.join(map(str, shape[2:]))}) on {device}; got {b!r}")
    return out


def _region_args(model, inputs, target, feature_mask, baselines, joint, internal_batch_size, who):
    """The argument checks of ``feature_ablation`` and ``shapley_sampling``, in order, before any launch.  Returns the towers,
    the per-tower baselines, the (B,) target rows, the int32 contiguous mask, F = max id + 1 and the fp32 inputs."""
    if not isinstance(joint, bool):
        raise ValueError(f"{who}: joint must be True or False; got {joint!r}")
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
    _refuse_tower_hooks(towers, who, "ablated")
    shape = tuple(inputs[0].shape)
    B, dims, dev = shape[0], shape[2:], inputs[0].device
    mask = feature_mask
    if (not torch.is_tensor(mask) or mask.is_floating_point() or mask.is_complex() or mask.dtype == torch.bool
            or mask.dim() != 5 or mask.shape[0] not in (1, B) or tuple(mask.shape[1:]) != shape[1:] or mask.device != dev):
        got = f"{mask.dtype} {tuple(mask.shape)} on {mask.device}" if torch.is_tensor(mask) else repr(mask)
        raise ValueError(f"{who}: feature_mask must be an integer tensor of shape (1|{B}, 1, {', '.join(map(str, dims))}) on "
                         f"{dev}; got {got}")
    bls = _ablation_baselines(baselines, len(towers), shape, dev, who)
    idx = _target_index(target, B, dev, who)
    if not all(x.is_cuda for x in inputs):
        raise ValueError(f"{who}: inputs must be CUDA tensors")
    lo, hi = (int(v) for v in torch.stack(mask.aminmax()).tolist())           # one device-to-host copy of the id range
    if lo < 0:
        raise ValueError(f"{who}: feature_mask ids must be >= 0; found {lo}")
    if hi >= 2 ** 31 - 1:
        raise ValueError(f"{who}: feature_mask ids must be below 2^31 - 1; found {hi}")
    F = hi + 1
    mask = mask.to(torch.int32).contiguous()
    xs = [TF._f32c(x.detach()) for x in inputs]
    return towers, bls, idx, mask, F, xs


def feature_ablation(model, inputs, target, feature_mask, baselines=0.0, joint=False, internal_batch_size=None):
    """Feature ablation over the regions of ``feature_mask`` through every sNet tower of ``model`` (eval mode), for the
    objective f = ``logits[b, target_b]`` of the model's first output (captum's ``FeatureAblation`` with a feature mask).

    ``feature_mask``: an integer tensor (1|B, 1, D, H, W) on the inputs' device; every id present, 0 included, is one feature,
    and ids must be >= 0.  It applies to every tower's input (the modalities are co-registered); a per-sample mask ablates
    each sample's own region.  ``baselines``: a finite Python scalar, or a tuple of one entry per tower, each a finite scalar
    or an fp32 CUDA tensor (1|B, 1, D, H, W); inside the feature the voxels take the baseline's value.  ``joint``: False
    ablates a feature in one tower's input at a time; True ablates it in every tower's input at once (captum's
    ``enable_cross_tensor_attribution``).  ``inputs``, ``target`` and ``internal_batch_size`` (volumes per pass) as for
    ``occlusion``.

    Returns ``FeatureAblation(maps, scores)``, per tower in tower order: ``scores`` fp32 (B, F), F = max id + 1, f(x) - f(x
    with feature j ablated) (0 for an id absent from the mask; with ``joint`` every tower has the same scores); ``maps`` fp32
    (B,1,D,H,W), each voxel holding its feature's score.

    The ablated towers are not run in full (DESIGN section 3.12): as in ``occlusion``, each feature recomputes only what its
    bounding box changes, on crops of one extent per extent class of features, and the composed tower outputs go through
    the model's own fusion stack and heads.  No parameter receives a ``.grad``, no weight-gradient kernel runs, BatchNorm
    buffers and the module mode are untouched and ``requires_grad`` flags are restored."""
    who = "feature_ablation"
    towers, bls, idx, mask, F, xs = _region_args(model, inputs, target, feature_mask, baselines, joint,
                                                 internal_batch_size, who)
    B, dims, dev = xs[0].shape[0], tuple(xs[0].shape[2:]), xs[0].device
    spec = towers[0]._spec
    layers = [(ks, pool) for _, _, ks, pool in spec.layers]
    boxes = TF.abl_boxes(mask, F)
    plans = [TF.abl_plan(boxes, ids, dims, layers) for _, ids in TF.abl_classes(boxes, dims)]
    groups = _tower_groups(towers)
    nt = len(towers)
    blocks = 1 if joint else nt

    flags = [(p, p.requires_grad) for p in model.parameters()]
    try:
        for p, _ in flags:
            p.requires_grad_(False)
        f_x, kept, base = _base_forward(model, towers, xs, idx, who)
        scores = torch.zeros((blocks, F, B), dtype=torch.float32, device=dev)
        for plan in plans:
            tabs = [torch.from_numpy(tb).to(dev) for tb in plan.tab]      # ordinary host-to-device copies
            fids = torch.from_numpy(plan.ids).to(dev)
            chunk = plan.n if internal_batch_size is None else max(1, internal_batch_size // B)
            chunk = min([chunk] + [TF.occ_pass_limit(plan, towers[g[0]]._spec, B, len(g)) for g in groups])
            for n0 in range(0, plan.n, chunk):
                m = min(chunk, plan.n - n0)
                # joint: every tower's rows 0 .. m*B are composed from its own crops; else rows [u*m*B, (u+1)*m*B) ablate
                # tower u, and the other towers' outputs there are replicated from their base outputs
                bufs = [torch.empty((blocks * m * B,) + plan.crop[-1] + (b.shape[-1],), dtype=torch.float32, device=dev)
                        for b in base]
                tab = [tb[n0:n0 + m] for tb in tabs]
                for grp in groups:
                    act = TF.abl_input([xs[t] for t in grp], mask, [bls[t] for t in grp], tab[0], fids[n0:n0 + m], m,
                                       plan.crop[0])
                    TF.occ_crops(towers[grp[0]]._spec, towers[grp[0]]._hyper(), [towers[t]._folds for t in grp], act,
                                 [kept[t] for t in grp], [base[t] for t in grp], plan, tab, m,
                                 [bufs[t][(0 if joint else t) * m * B:((0 if joint else t) + 1) * m * B] for t in grp])
                f_abl = _through_fusion(model, towers, xs, base, bufs, tab[-1], m, plan.crop[-1], idx, blocks)
                scores[:, plan.ids[n0:n0 + m].tolist()] = f_x.view(1, 1, B) - f_abl
    finally:
        for p, f in flags:
            p.requires_grad_(f)
        for t in towers:
            t._lrp_keep = None
            t._occ_out = None
    per = [s.t().contiguous() for s in scores.unbind(0)]
    if joint:
        per += [per[0].clone() for _ in range(nt - 1)]
    return FeatureAblation(TF.abl_map(per, mask), per)


ShapleySampling = namedtuple("ShapleySampling", ["maps", "scores", "delta", "permutations"])


def shapley_sampling(model, inputs, target, feature_mask, baselines=0.0, joint=False, n_samples=25,
                     internal_batch_size=None):
    """Shapley value sampling (Castro, Gomez & Tejada, 2009; Strumbelj & Kononenko, 2014) over the regions of
    ``feature_mask`` through every sNet tower of ``model`` (eval mode), for the objective f = ``logits[b, target_b]`` of the
    model's first output (captum's ``ShapleyValueSampling`` with a feature mask).

    The players are the ids present in the mask, 0 included.  ``n_samples`` permutations of them are drawn with
    ``torch.randperm`` from torch's global CPU generator, one per sample draw, shared by all B samples and every tower.  A
    chain walks one permutation from the start state -- the baseline everywhere in the ablated input(s) -- to x: step k sets
    the voxels of region pi[k] to x, and its marginal contribution is f(after) - f(before); a region's score is the mean of its
    contributions over the permutations (positive: the region's real values raise the target logit).  ``joint``: False plays
    one game per tower (only tower t's input walks, the others see x); True plays one game in which a region enters every
    tower's input at once, and every tower reports its scores.  ``inputs``, ``target``, ``feature_mask``, ``baselines`` and
    ``internal_batch_size`` (volumes per pass; it changes the speed only, never the bits) as for ``feature_ablation``.

    Returns ``ShapleySampling(maps, scores, delta, permutations)``, per tower in tower order: ``scores`` fp32 (B, F), F = max
    id + 1 (0 for an id absent from the mask); ``maps`` fp32 (B,1,D,H,W), each voxel holding its region's score; ``delta`` fp32
    (B,), sum_j scores[:, j] - (f(x) - f(start)).  The contributions of a chain telescope, so delta is only the rounding of
    the recomputation, never sampling error.  ``permutations``: int64 (n_samples, F'), the orders of the F' present ids used.

    The towers are not run per step (DESIGN section 3.13): each chain keeps its own copy of every layer's input activation,
    and a step recomputes only the added region's bounding box on the crops of ``feature_ablation``, writing the result back
    into the chain's copy.  No parameter receives a ``.grad``, no weight-gradient kernel runs, BatchNorm buffers and the
    module mode are untouched and ``requires_grad`` flags are restored."""
    import numpy as np
    who = "shapley_sampling"
    if not _is_count(n_samples):
        raise ValueError(f"{who}: n_samples must be an integer >= 1; got {n_samples!r}")
    towers, bls, idx, mask, F, xs = _region_args(model, inputs, target, feature_mask, baselines, joint,
                                                 internal_batch_size, who)
    B, dims, dev = xs[0].shape[0], tuple(xs[0].shape[2:]), xs[0].device
    spec = towers[0]._spec
    layers = [(ks, pool) for _, _, ks, pool in spec.layers]
    boxes = TF.abl_boxes(mask, F)
    classes = TF.abl_classes(boxes, dims)
    plans = [TF.abl_plan(boxes, ids, dims, layers) for _, ids in classes]
    cls_of = {f: c for c, (_, ids) in enumerate(classes) for f in ids}
    row_of = {f: n for plan in plans for n, f in enumerate(plan.ids.tolist())}
    players = np.array(sorted(cls_of), dtype=np.int64)
    perms = TF.shap_permutations(players, n_samples)
    P, Fp = perms.shape
    pn = perms.numpy()
    rank = np.full((P, F), np.iinfo(np.int32).max, dtype=np.int32)
    rank[np.arange(P)[:, None], pn] = np.arange(Fp, dtype=np.int32)
    groups = _tower_groups(towers)
    nt = len(towers)
    blocks = 1 if joint else nt
    chunk = P if internal_batch_size is None else max(1, internal_batch_size // B)
    caps = [min([chunk] + [TF.occ_pass_limit(plan, towers[g[0]]._spec, B, len(g)) for g in groups]) for plan in plans]

    flags = [(p, p.requires_grad) for p in model.parameters()]
    try:
        for p, _ in flags:
            p.requires_grad_(False)
        f_x, _, base = _base_forward(model, towers, xs, idx, who)
        starts = [torch.full_like(x, b) if not torch.is_tensor(b) else b.expand_as(x).contiguous() for x, b in zip(xs, bls)]
        _, kept, start_out = _base_forward(model, towers, starts, idx, who)
        # f(start) through the fusion stack as the passes run it: block u holds tower u's start output (joint: every tower's)
        zero_tab = torch.zeros((1, 3, 4), dtype=torch.int32, device=dev)
        bufs = [torch.empty((blocks * B,) + tuple(b.shape[1:]), dtype=torch.float32, device=dev) for b in base]
        for t in range(nt):
            bufs[t][(0 if joint else t) * B:((0 if joint else t) + 1) * B].copy_(start_out[t])
        f_start = _through_fusion(model, towers, xs, base, bufs, zero_tab, 1, tuple(base[0].shape[1:4]), idx, blocks)[:, 0]
        # f along every chain: fv[:, p, k] after step k - 1 of chain p (k = 0: the start state)
        fv = torch.empty((blocks, P, Fp + 1, B), dtype=torch.float32, device=dev)
        fv[:, :, 0] = f_start.unsqueeze(1)
        per_chain = sum(sum(k[l][0].nbytes for l in range(1, len(k))) + o.nbytes for k, o in zip(kept, start_out))
        Pg = max(1, min(P, TF.SHAP_STATE_BYTES // per_chain))
        rank_d = torch.from_numpy(rank).to(dev)                                # ordinary host-to-device copies
        chain, region = torch.arange(P).repeat_interleave(Fp).to(dev), perms.reshape(-1).to(dev)
        for p0 in range(0, P, Pg):
            S = min(Pg, P - p0)
            # every chain starts from the start state: (S*B, ...) copies of the kept layer inputs and the tower output
            state = [[None] + [a.repeat((S,) + (1,) * (a.dim() - 1)) for a in [kl[0] for kl in k[1:]] + [o]]
                     for k, o in zip(kept, start_out)]
            passes = TF.shap_schedule(pn[p0:p0 + S], cls_of, caps)
            rows = [(c, p, k) for c, steps in passes for p, k in steps]
            n_at = [row_of[int(pn[p0 + p, k])] for _, p, k in rows]
            tab_all = [torch.from_numpy(np.stack([plans[c].tab[l][n] for (c, _, _), n in zip(rows, n_at)])).to(dev)
                       for l in range(len(layers) + 1)]
            meta = torch.from_numpy(np.array([[p0 + p, k, p] for _, p, k in rows], dtype=np.int32).T.copy()).to(dev)
            at_all = torch.tensor([(p0 + p) * (Fp + 1) + k + 1 for _, p, k in rows], dtype=torch.int64).to(dev)
            r0 = 0
            for c, steps in passes:
                m, plan = len(steps), plans[c]
                assert len({p for p, _ in steps}) == m                           # a chain at most once per pass
                perm, step, sidx = (v[r0:r0 + m] for v in meta)
                tab = [tb[r0:r0 + m] for tb in tab_all]
                bufs = [torch.empty((blocks * m * B,) + plan.crop[-1] + (b.shape[-1],), dtype=torch.float32, device=dev)
                        for b in base]
                for grp in groups:
                    act = TF.shap_input([xs[t] for t in grp], mask, [bls[t] for t in grp], tab[0], rank_d, perm, step, m,
                                        plan.crop[0])
                    TF.shap_crops(towers[grp[0]]._spec, towers[grp[0]]._hyper(), [towers[t]._folds for t in grp], act,
                                  [state[t] for t in grp], plan, tab, sidx, m,
                                  [bufs[t][(0 if joint else t) * m * B:((0 if joint else t) + 1) * m * B] for t in grp])
                f_new = _through_fusion(model, towers, xs, base, bufs, tab[-1], m, plan.crop[-1], idx, blocks)
                fv.view(blocks, P * (Fp + 1), B)[:, at_all[r0:r0 + m]] = f_new
                r0 += m
            del state
    finally:
        for p, f in flags:
            p.requires_grad_(f)
        for t in towers:
            t._lrp_keep = None
            t._occ_out = None
    contrib = torch.zeros((blocks, P, F, B), dtype=torch.float32, device=dev)
    contrib[:, chain, region] = (fv[:, :, 1:] - fv[:, :, :-1]).reshape(blocks, P * Fp, B)
    total = contrib[:, 0].clone()
    for p in range(1, P):                                                     # a fixed order, whatever the grouping
        total += contrib[:, p]
    scores = [s.t().contiguous() for s in (total / P).unbind(0)]
    delta = [s.sum(1) - (f_x - fs) for s, fs in zip(scores, f_start.unbind(0))]
    if joint:
        scores += [scores[0].clone() for _ in range(nt - 1)]
        delta += [delta[0].clone() for _ in range(nt - 1)]
    return ShapleySampling(TF.abl_map(scores, mask), scores, delta, perms)
