"""Building blocks of TransMF_AD on the B200 kernels -- drop-in for the reference ``models/networks.py``.

Every class keeps the reference's name, constructor signature, sub-module names (hence ``state_dict`` keys, shapes and
fp32 dtype) and forward signature; the torch ``nn.Conv3d`` / ``nn.BatchNorm3d`` / ``nn.Linear`` / ``nn.LayerNorm``
children are *parameter containers only* -- their forward is never called.  All arithmetic goes through
``transmf_ad_b200.functional`` (C ABI -> sm_100a kernels).  Reference line numbers are cited per class.
"""
from __future__ import annotations

import contextlib
import copy
import warnings
import weakref

import torch
from torch import nn

from transmf_ad_b200 import functional as TF


def exists(val):
    return val is not None


def default(val, d):
    return val if exists(val) else d


# ---------------------------------------------------------------------------------------------------------------
# 3D-CNN encoder   (reference models/networks.py:18-61)
# ---------------------------------------------------------------------------------------------------------------
def _conv_unit(cin, cout, k):
    return [nn.Conv3d(cin, cout, kernel_size=(k, k, k), padding=k // 2), nn.BatchNorm3d(cout), nn.LeakyReLU()]


class sNet(nn.Module):
    """7x(Conv3d + BatchNorm3d + LeakyReLU) with three MaxPool3d(2,2) and a final AvgPool3d(2,2)."""

    def __init__(self, dim) -> None:
        super().__init__()
        q, h = dim // 4, dim // 2
        self.conv1 = nn.Sequential(*_conv_unit(1, q, 3), nn.MaxPool3d(2, stride=2))
        self.conv2 = nn.Sequential(*_conv_unit(q, q, 3), *_conv_unit(q, h, 3), nn.MaxPool3d(2, stride=2))
        self.conv3 = nn.Sequential(*_conv_unit(h, h, 3), *_conv_unit(h, dim, 3), nn.MaxPool3d(2, stride=2))
        self.conv4 = nn.Sequential(*_conv_unit(dim, dim * 2, 3), *_conv_unit(dim * 2, dim, 1), nn.AvgPool3d(2, stride=2))
        self._spec = TF.SNetSpec(dim)
        self._packs = [TF.ConvPack() for _ in range(7)]      # cached bf16 operand packs of the conv weights
        self._folds = [TF.EvalFold() for _ in range(7)]      # eval mode: BatchNorm folded into the conv operands
        self._cam_tap = None                                  # transmf_ad_b200.interpret.grad_cam: block index to expose
        self._cam_act = None
        self._lrp_keep = None          # transmf_ad_b200.interpret.lrp: a list the folded eval forward appends (a, y) to
        self._lrp_folds = {}           # LRP rule -> 7 TF.LrpFold
        self._ig_src = None            # transmf_ad_b200.interpret.integrated_gradients: block 1's output (fp32 leaf, bf16 twin)
        self._occ_out = None           # transmf_ad_b200.interpret.occlusion: the composed tower output, returned as is

    def _units(self):
        """[(conv, bn)] in execution order."""
        return [(self.conv1[0], self.conv1[1]), (self.conv2[0], self.conv2[1]), (self.conv2[3], self.conv2[4]),
                (self.conv3[0], self.conv3[1]), (self.conv3[3], self.conv3[4]), (self.conv4[0], self.conv4[1]),
                (self.conv4[3], self.conv4[4])]

    def _hyper(self):
        """Per layer (eps, momentum, negative_slope) read from the BatchNorm3d / LeakyReLU children."""
        seqs = [(self.conv1, 0), (self.conv2, 0), (self.conv2, 3), (self.conv3, 0), (self.conv3, 3), (self.conv4, 0),
                (self.conv4, 3)]
        out = []
        for seq, i in seqs:
            bn, act = seq[i + 1], seq[i + 2]
            if bn.momentum is None or not bn.track_running_stats or not bn.affine:
                raise NotImplementedError("sNet on the B200 kernels needs affine BatchNorm3d with running statistics and "
                                          "a numeric momentum (the reference's nn.BatchNorm3d defaults)")
            if not act.negative_slope >= 0:
                raise NotImplementedError("sNet on the B200 kernels needs LeakyReLU slopes >= 0: the max pools route gradients "
                                          f"by the pre-BatchNorm value, which a negative slope reorders (got {act.negative_slope})")
            out.append((float(bn.eps), float(bn.momentum), float(act.negative_slope)))
        return out

    def _run(self, other=None):
        packs = [self._packs] if other is None else [self._packs, other._packs]
        folds = [self._folds] if other is None else [self._folds, other._folds]
        # torch.nn.SyncBatchNorm.convert_sync_batchnorm(model) turns the BatchNorm3d children into nn.SyncBatchNorm: the kernels
        # then normalise with statistics over the global batch (SURVEY.md section 8e, optional row)
        sync = [isinstance(bn, nn.SyncBatchNorm) for _, bn in self._units()]
        if any(sync) and not all(sync):
            raise NotImplementedError("sNet: either every BatchNorm3d is an nn.SyncBatchNorm or none")
        group = self._units()[0][1].process_group if all(sync) else False
        keep = [self._lrp_keep] if other is None else [self._lrp_keep, other._lrp_keep]
        return TF.SNetRun(self.training, torch.is_grad_enabled(), self._hyper(), packs, folds, sync_group=group,
                          keep=keep if any(k is not None for k in keep) else None)

    def invalidate_packs(self):
        for pk in self._packs:
            pk.version = None

    def pack_now(self):
        """(Re-)pack every conv weight now, e.g. after weights were restored outside an optimizer step, so that a CUDA-graph
        capture that follows contains no pack launches (``optim.FusedAdam`` keeps the packs fresh from then on)."""
        from transmf_ad_b200 import _lib as L
        for l, (conv, _) in enumerate(self._units()):
            if l == 0 or not conv.weight.is_cuda:
                continue
            pk, w = self._packs[l], conv.weight
            pk.stale(w)
            L.call("tmf_pack_conv_weights", 1, L.ptrs([w.detach()]), L.ptrs([pk.wf]), L.ptrs([pk.wd]), w.shape[0], w.shape[1],
                   w.shape[2])
            pk.mark(w)

    def _params_and_buffers(self):
        params, bufs = [], []
        for conv, bn in self._units():
            params += [conv.weight, conv.bias, bn.weight, bn.bias]
            bufs.append((bn.running_mean, bn.running_var, bn.num_batches_tracked))
        return params, bufs

    def forward(self, mri):
        if self._occ_out is not None:
            return self._occ_out
        params, bufs = self._params_and_buffers()
        taps = _tapped_boundaries([self])
        if taps:
            return _segmented_forward([self], [mri], params, [bufs], taps)[0]
        return TF.SNetFunction.apply(self._spec, self._run(), [bufs], 1, mri, *params)


def snet_pair_forward(net_a: sNet, net_b: sNet, xa, xb):
    """Run two towers of identical shape as one grouped launch sequence (grid.z = tower).  Forward pre-hooks and forward
    hooks of the towers fire as ``nn.Module.__call__`` would fire them; towers with backward hooks go through it."""
    if (net_a._occ_out is not None or net_b._occ_out is not None
            or net_a._spec.dim != net_b._spec.dim or net_a.training != net_b.training or tuple(xa.shape) != tuple(xb.shape)
            or net_a._hyper() != net_b._hyper() or _has_backward_hooks(net_a) or _has_backward_hooks(net_b)):
        return net_a(xa), net_b(xb)
    xa, xb = _fire_pre_hooks(net_a, xa), _fire_pre_hooks(net_b, xb)
    pa, ba = net_a._params_and_buffers()
    pb, bb = net_b._params_and_buffers()
    taps = _tapped_boundaries([net_a, net_b])
    if taps:
        fa, fb = _segmented_forward([net_a, net_b], [xa, xb], pa + pb, [ba, bb], taps)
    else:
        fa, fb = TF.SNetFunction.apply(net_a._spec, net_a._run(net_b), [ba, bb], 2, xa, xb, *pa, *pb)
    return _fire_hooks(net_a, xa, fa), _fire_hooks(net_b, xb, fb)


# ---------------------------------------------------------------------------------------------------------------
# block outputs for module hooks and Grad-CAM   (DESIGN section 3.7)
# ---------------------------------------------------------------------------------------------------------------
BLOCKS = ("conv1", "conv2", "conv3", "conv4")
BLOCK_END = (0, 2, 4, 6)              # last sNet layer of each block; boundary k = output of block k (3: the tower output)
_WARNED = weakref.WeakSet()


def _has_backward_hooks(m):
    return bool(m._backward_hooks or m._backward_pre_hooks)


def _fire_pre_hooks(m, x, block=False):
    """``nn.Module.__call__``'s forward pre-hooks on the single positional argument x; a block's hooks may only observe."""
    for hid, hook in list(m._forward_pre_hooks.items()):
        if hid in m._forward_pre_hooks_with_kwargs:
            res = hook(m, (x,), {})
            res = None if res is None else res[0]
        else:
            res = hook(m, (x,))
        if res is not None:
            if block:
                raise NotImplementedError(f"a forward pre-hook on sNet.{_block_name(m)} returned a replacement input: the block "
                                          f"runs inside fused kernels, so its hooks may only observe")
            x = res[0] if isinstance(res, tuple) else res
    return x


def _fire_hooks(m, x, out, block=False):
    """``nn.Module.__call__``'s forward hooks with (module, (x,), out); a block's hooks may only observe."""
    for hid, hook in list(m._forward_hooks.items()):
        res = hook(m, (x,), {}, out) if hid in m._forward_hooks_with_kwargs else hook(m, (x,), out)
        if res is not None:
            if block:
                raise NotImplementedError(f"a forward hook on sNet.{_block_name(m)} returned a replacement output: the block "
                                          f"runs inside fused kernels, so its hooks may only observe")
            out = res
    return out


def _block_name(m):
    return getattr(m, "_tmf_block_name", "conv?")


def _tapped_boundaries(nets):
    """Block outputs the hooks on the towers' blocks (and a pending Grad-CAM) need as real tensors: a hook on block k taps
    its input (boundary k-1) and its output (boundary k).  Refuses what cannot be honoured and warns, once per module, about
    hooks on modules inside a block (their tensors are fused away and never exist)."""
    taps = set()
    for net in nets:
        if net._cam_tap is not None:
            taps.add(net._cam_tap)
        if net._ig_src is not None:
            taps.add(0)
        for k, name in enumerate(BLOCKS):
            blk = getattr(net, name)
            if _has_backward_hooks(blk):
                raise NotImplementedError(f"backward hooks on sNet.{name} are not supported (the block runs inside fused "
                                          f"kernels): register a tensor hook on its output from a forward hook "
                                          f"(output.register_hook) or use torch.autograd.grad with respect to that output")
            if blk._forward_hooks or blk._forward_pre_hooks:
                blk._tmf_block_name = name
                taps.update((k - 1, k) if k > 0 else (k,))
            for child in blk._modules.values():
                if (child._forward_hooks or child._forward_pre_hooks or _has_backward_hooks(child)) and child not in _WARNED:
                    _WARNED.add(child)
                    warnings.warn(f"a hook on {type(child).__name__} inside sNet.{name} never fires: the block's layers run "
                                  f"as fused kernels and their intermediate tensors do not exist. Hook the blocks "
                                  f"({', '.join(BLOCKS)}) or the sNet itself", UserWarning, stacklevel=4)
    return taps


def segment_plan(taps):
    """Layer ranges [(l0, l1)] of a segmented run: split after each tapped block (the tower output is always exposed)."""
    cuts = sorted(BLOCK_END[k] + 1 for k in taps if k < len(BLOCKS) - 1) + [BLOCK_END[-1] + 1]
    return list(zip([0] + cuts[:-1], cuts))


def _segmented_forward(nets, xs, params, bufs, taps):
    """The towers as a chain of ``SNetFunction`` nodes split after every tapped block: each block output is an fp32 tensor
    on the autograd path (its bf16 twin feeds the next segment), and the blocks' hooks fire on it."""
    spec, ng = nets[0]._spec, len(nets)
    run = nets[0]._run(nets[1] if ng == 2 else None)
    cam = nets[0]._cam_tap
    if cam is not None:
        # Grad-CAM: everything up to the exposed block runs without autograd (no backward launches upstream of it)
        run_nograd = copy.copy(run)
        run_nograd.grad_enabled = False
    cuts = [l1 for _, l1 in segment_plan(taps)]
    bound = {-1: list(xs)}
    supplied = [net._ig_src for net in nets]
    if any(s is not None for s in supplied):
        # integrated gradients supplies block 1's output for every path point: the towers start at layer 1 and the
        # volumes xs are never read
        if any(s is None for s in supplied):
            raise RuntimeError("a block-1 output was supplied for only one tower of a pair")
        cur, src, l0 = [s[0] for s in supplied], [s[1] for s in supplied], BLOCK_END[0] + 1
        bound[0] = cur
        cuts = cuts[1:]
        for t, net in enumerate(nets):
            if net.conv2._forward_pre_hooks:
                _fire_pre_hooks(net.conv2, cur[t], block=True)
    else:
        for t, net in enumerate(nets):
            if net.conv1._forward_pre_hooks:
                _fire_pre_hooks(net.conv1, xs[t], block=True)
        cur, src, l0 = list(xs), None, 0
    for l1 in cuts:
        upstream = cam is not None and l1 <= BLOCK_END[cam] + 1
        with torch.no_grad() if upstream else contextlib.nullcontext():
            res = TF.SNetFunction.apply(TF.SNetSegment(spec, l0, l1, src), run_nograd if upstream else run, bufs, ng,
                                        *cur, *params)
        res = res if isinstance(res, tuple) else (res,)
        k = BLOCK_END.index(l1 - 1)
        outs, src = list(res[:ng]), list(res[ng:]) or None
        if cam == k:
            outs = [o.detach().requires_grad_(True) for o in outs]
            for net, o in zip(nets, outs):
                net._cam_act = o
        bound[k] = outs
        versions = [o._version for o in outs]
        for t, net in enumerate(nets):
            blk = getattr(net, BLOCKS[k])
            if blk._forward_hooks:
                _fire_hooks(blk, bound[k - 1][t], outs[t], block=True)
            if k + 1 < len(BLOCKS) and getattr(net, BLOCKS[k + 1])._forward_pre_hooks:
                _fire_pre_hooks(getattr(net, BLOCKS[k + 1]), outs[t], block=True)
        if src is not None and [o._version for o in outs] != versions:
            raise RuntimeError(f"a hook modified the output of sNet.{BLOCKS[k]} in place; the next block would read the "
                               f"value from before the change. Hooks on sNet blocks may only observe (clone to modify)")
        cur, l0 = outs, l1
    return cur


def tokens_of(feat):
    """'b d x y z -> b (x y z) d' (reference models/mymodel.py:218-219); a free view of the channels-last output."""
    B, C = feat.shape[:2]
    return feat.permute(0, 2, 3, 4, 1).reshape(B, -1, C)


# ---------------------------------------------------------------------------------------------------------------
# transformer blocks   (reference models/networks.py:114-175, 215-230)
# ---------------------------------------------------------------------------------------------------------------
class Linear(nn.Linear):
    """nn.Linear whose forward is the tmf GEMM kernel (same parameters / state_dict keys)."""

    def forward(self, x):
        return TF.linear(x, self.weight, self.bias)


def _dropout_active(mod):
    return mod.training and mod.p > 0


class PreNorm(nn.Module):
    """LayerNorm on the first argument only; ``context`` passes through raw (reference :114-121)."""

    def __init__(self, dim, fn):
        super().__init__()
        self.norm = nn.LayerNorm(dim)
        self.fn = fn

    def forward(self, x, **kwargs):
        return self.fn(TF.layer_norm(x, self.norm.weight, self.norm.bias, eps=self.norm.eps), **kwargs)


class FeedForward(nn.Module):
    """Linear - exact GELU - Dropout - Linear - Dropout (reference :125-137)."""

    def __init__(self, dim, hidden_dim, dropout=0.):
        super().__init__()
        self.net = nn.Sequential(nn.Linear(dim, hidden_dim), nn.GELU(), nn.Dropout(dropout),
                                 nn.Linear(hidden_dim, dim), nn.Dropout(dropout))

    def forward(self, x, residual=None):
        h = TF.linear(x, self.net[0].weight, self.net[0].bias, gelu=True)
        if _dropout_active(self.net[2]):
            h = self.net[2](h)
        if _dropout_active(self.net[4]):
            y = self.net[4](TF.linear(h, self.net[3].weight, self.net[3].bias))
            return y if residual is None else y + residual
        return TF.linear(h, self.net[3].weight, self.net[3].bias, residual=residual)


class Attention(nn.Module):
    """Multi-head (cross-)attention, bias-free q / kv projections (reference :141-175)."""

    def __init__(self, dim, heads=4, dim_head=64, dropout=0.):
        super().__init__()
        inner_dim = dim_head * heads
        self.heads = heads
        self.scale = dim_head ** -0.5
        self.attend = nn.Softmax(dim=-1)
        self.to_q = nn.Linear(dim, inner_dim, bias=False)
        self.to_kv = nn.Linear(dim, inner_dim * 2, bias=False)
        self.to_out = nn.Sequential(nn.Linear(inner_dim, dim), nn.Dropout(dropout))

    def forward(self, x, context=None, kv_include_self=False, residual=None):
        context = default(context, x)
        if kv_include_self:
            context = torch.cat((x, context), dim=1)
        q = TF.linear(x, self.to_q.weight)
        kv = TF.linear(context, self.to_kv.weight)
        if _attend_hooked(self.attend):
            tap = TF.AttnTap()
            out, dots, attn = TF.attention_core(q, kv, self.heads, self.scale, tap)
            out = TF.attn_tap(out, attn, tap)
            _fire_attend_hooks(self.attend, dots, attn)
        else:
            out = TF.attention_core(q, kv, self.heads, self.scale)
        proj, drop = self.to_out[0], self.to_out[1]
        if _dropout_active(drop):
            y = drop(TF.linear(out, proj.weight, proj.bias))
            return y if residual is None else y + residual
        return TF.linear(out, proj.weight, proj.bias, residual=residual)


class Transformer(nn.Module):
    """depth x (pre-LN attention + pre-LN FFN, each with a residual) and a trailing LayerNorm (reference :215-230)."""

    def __init__(self, dim, depth, heads, dim_head, mlp_dim, dropout=0.):
        super().__init__()
        self.layers = nn.ModuleList([])
        self.norm = nn.LayerNorm(dim)
        self._enc_pack = TF.EncPack()          # cached bf16 hi / lo operand pack of the fused encoder (depth 1)
        for _ in range(depth):
            self.layers.append(nn.ModuleList([
                PreNorm(dim, Attention(dim, heads=heads, dim_head=dim_head, dropout=dropout)),
                PreNorm(dim, FeedForward(dim, mlp_dim, dropout=dropout))]))

    def _enc_weights(self):
        attn, ff = self.layers[0]
        return (attn.fn.to_q.weight, attn.fn.to_kv.weight, attn.fn.to_out[0].weight, ff.fn.net[0].weight, ff.fn.net[3].weight)

    def invalidate_packs(self):
        self._enc_pack.versions = {}

    def pack_now(self):
        """(Re-)pack the five weight matrices now (see ``sNet.pack_now``): a CUDA-graph capture that follows then contains no
        ``tmf_encoder_pack_weights`` launch; ``optim.FusedAdam`` keeps the pack fresh from its own kernel."""
        from transmf_ad_b200 import _lib as L
        ws = self._enc_weights()
        if len(self.layers) != 1 or not ws[0].is_cuda or not TF.encoder_supported(ws[0].shape[1], ws[0].shape[0], ws[3].shape[0]):
            return
        pk = self._enc_pack
        pk.stale(ws, ws[3].shape[0])
        L.call("tmf_encoder_pack_weights", *[L.ptr(w.detach()) for w in ws], int(ws[3].shape[0]), L.ptr(pk.pack))
        for w in ws:
            pk.mark(w)

    def _fused_params(self):
        attn, ff = self.layers[0]
        A, F = attn.fn, ff.fn
        return (attn.norm.weight, attn.norm.bias, A.to_q.weight, A.to_kv.weight, A.to_out[0].weight, A.to_out[0].bias,
                ff.norm.weight, ff.norm.bias, F.net[0].weight, F.net[0].bias, F.net[3].weight, F.net[3].bias,
                self.norm.weight, self.norm.bias)

    def _can_fuse(self, x, context):
        if len(self.layers) != 1 or context is None or x.dim() != 3 or context.dim() != 3 or not x.is_cuda:
            return False
        attn, ff = self.layers[0]
        A, F = attn.fn, ff.fn
        if _dropout_active(A.to_out[1]) or _dropout_active(F.net[2]) or _dropout_active(F.net[4]):
            return False
        dim = x.shape[-1]
        return (A.to_out[0].bias is not None and F.net[0].bias is not None and F.net[3].bias is not None and
                TF.encoder_supported(dim, A.to_q.weight.shape[0], F.net[0].weight.shape[0]) and context.shape[-1] == dim)

    def _dead_hook_scan(self, fused):
        """Warn, once per module, about hooks on children whose forward never runs: the nn.Linear / nn.LayerNorm / nn.GELU
        parameter containers, an inactive nn.Dropout and, on the fused path, PreNorm / Attention / FeedForward as well."""
        for pair in self.layers:
            for pre in pair:
                mods = [pre.norm, *pre.fn.children()] + (list(pre.fn.net) if isinstance(pre.fn, FeedForward) else
                                                         list(pre.fn.to_out))
                if fused:
                    mods += [pre, pre.fn]
                for m in mods:
                    if m is getattr(pre.fn, "attend", None):
                        continue
                    if isinstance(m, nn.Dropout) and not fused and _dropout_active(m):
                        continue
                    _warn_dead_hook(m)
        _warn_dead_hook(self.norm)

    def forward(self, x, context=None, add_input=False):
        """``add_input`` fuses the caller's outer residual ``enc(x) + x`` into the final LayerNorm kernel."""
        if self._can_fuse(x, context):
            attn, ff = self.layers[0]          # the whole encoder in 3 launches (csrc/enc_fused.cu)
            self._dead_hook_scan(True)
            tap = TF.AttnTap() if _attend_hooked(attn.fn.attend) else None
            y = TF.encoder(x, context, attn.fn.heads, attn.fn.scale, add_input, attn.norm.eps, ff.norm.eps,
                           self.norm.eps, self._fused_params(), pack_cache=self._enc_pack, tap=tap)
            if tap is None:
                return y
            y, dots, probs = y
            y = TF.attn_tap(y, probs, tap)
            _fire_attend_hooks(attn.fn.attend, dots, probs)
            return y
        self._dead_hook_scan(False)
        x_in = x
        for attn, ff in self.layers:
            x = attn(x, context=context, residual=x)
            x = ff(x, residual=x)
        return TF.layer_norm(x, self.norm.weight, self.norm.bias, residual=x_in if add_input else None,
                             eps=self.norm.eps)


# ---------------------------------------------------------------------------------------------------------------
# attention probabilities for module hooks and attention maps   (DESIGN section 3.8)
# ---------------------------------------------------------------------------------------------------------------
def _attend_hooked(attend):
    """Whether ``Attention.attend`` has hooks to fire: the attention node then also returns ``dots`` / ``attn``."""
    if _has_backward_hooks(attend):
        raise NotImplementedError("backward hooks on Attention.attend are not supported (the softmax runs inside fused "
                                  "kernels): register a tensor hook on `attn` from a forward hook (attn.register_hook), "
                                  "or use torch.autograd.grad with respect to it")
    return bool(attend._forward_hooks or attend._forward_pre_hooks)


def _warn_dead_hook(m):
    if (m._forward_hooks or m._forward_pre_hooks or _has_backward_hooks(m)) and m not in _WARNED:
        _WARNED.add(m)
        warnings.warn(f"a hook on {type(m).__name__} inside a fusion Transformer never fires: the encoder runs as fused "
                      f"kernels and this module's forward is never called. Hook the attention probabilities at "
                      f"Attention.attend, or the Transformer itself", UserWarning, stacklevel=5)


def _fire_attend_hooks(attend, dots, attn):
    """``nn.Module.__call__``'s hooks of the reference's ``attn = self.attend(dots)``: pre-hooks get (dots,), forward hooks
    (module, (dots,), attn); they may only observe."""
    versions = (dots._version, attn._version)
    for hid, hook in list(attend._forward_pre_hooks.items()):
        res = hook(attend, (dots,), {}) if hid in attend._forward_pre_hooks_with_kwargs else hook(attend, (dots,))
        if res is not None:
            raise NotImplementedError("a forward pre-hook on Attention.attend returned a replacement input: the softmax "
                                      "runs inside fused kernels, so its hooks may only observe")
    for hid, hook in list(attend._forward_hooks.items()):
        res = hook(attend, (dots,), {}, attn) if hid in attend._forward_hooks_with_kwargs else hook(attend, (dots,), attn)
        if res is not None:
            raise NotImplementedError("a forward hook on Attention.attend returned a replacement output: the softmax runs "
                                      "inside fused kernels, so its hooks may only observe")
    if (dots._version, attn._version) != versions:
        raise RuntimeError("a hook modified the attention scores or probabilities in place; the model used the values "
                           "from before the change. Hooks on Attention.attend may only observe (clone to modify)")


class _TokenGAP(nn.Module):
    """'b n d -> b d' mean over tokens (reference :264-266)."""

    def forward(self, x):
        return TF.token_pool(x, True, False)


class _TokenGMP(nn.Module):
    """'b n d -> b d' max over tokens (reference :267-269)."""

    def forward(self, x):
        return TF.token_pool(x, False, True)


def _encoder_pairs(dim, depth, heads, dim_head, mlp_dim, dropout):
    return nn.ModuleList([nn.ModuleList([Transformer(dim, 1, heads, dim_head, mlp_dim, dropout=dropout),
                                         Transformer(dim, 1, heads, dim_head, mlp_dim, dropout=dropout)])
                          for _ in range(depth)])


class CrossTransformer(nn.Module):
    """Both encoders attend to cat([mri, pet]) (reference :233-252; ``share=True`` is broken upstream and unused)."""

    def __init__(self, dim, depth, heads, dim_head, mlp_dim, dropout, share=False):
        super().__init__()
        self.share = share
        if share:
            self.layers = nn.ModuleList([Transformer(dim, 1, heads, dim_head, mlp_dim, dropout=dropout)
                                         for _ in range(depth)])
        else:
            self.layers = _encoder_pairs(dim, depth, heads, dim_head, mlp_dim, dropout)

    def forward(self, mri_tokens, pet_tokens):
        for mri_enc, pet_enc in self.layers:
            mri_tokens = mri_enc(mri_tokens, context=torch.cat([mri_tokens, pet_tokens], dim=1), add_input=True)
            pet_tokens = pet_enc(pet_tokens, context=torch.cat([mri_tokens, pet_tokens], dim=1), add_input=True)
        return mri_tokens, pet_tokens


class CrossTransformer_MOD_AVG(nn.Module):
    """MRI attends to PET, then PET to the UPDATED MRI, ``depth`` times; cat[GAP mri, GAP pet, GMP mri, GMP pet]
    (reference :255-281)."""

    def __init__(self, dim, depth, heads, dim_head, mlp_dim, dropout):
        super().__init__()
        self.layers = _encoder_pairs(dim, depth, heads, dim_head, mlp_dim, dropout)
        self.gap = _TokenGAP()
        self.gmp = _TokenGMP()

    def forward(self, mri_tokens, pet_tokens):
        for mri_enc, pet_enc in self.layers:
            mri_tokens = mri_enc(mri_tokens, context=pet_tokens, add_input=True)
            pet_tokens = pet_enc(pet_tokens, context=mri_tokens, add_input=True)
        mri_avg, mri_max = TF.token_pool(mri_tokens, True, True)
        pet_avg, pet_max = TF.token_pool(pet_tokens, True, True)
        return torch.cat([mri_avg, pet_avg, mri_max, pet_max], dim=1)
