"""Host-side operators: thin wrappers over the C ABI (include/tmf.h) plus the ``torch.autograd.Function``s that
give the reference's ``nn.Module``s their forward and backward on the B200 kernels.

Nothing here computes on the CPU or through a torch library kernel on the hot path: tensors are allocated with
torch (caching allocator), every arithmetic op is a ``tmf_*`` launch on the current CUDA stream.
"""
from __future__ import annotations

import os

import torch

from . import _lib as L

BN_EPS, BN_MOMENTUM, LRELU_SLOPE, LN_EPS = 1e-5, 0.1, 0.01, 1e-5


# Data parallelism (dp.FlatGradReducer.install): parameter data_ptr -> (slot view of the flat gradient buffer, parameter).
# The backward kernels write weight gradients straight into the slots, autograd adopts the view as ``.grad`` without a
# copy, and the gradient exchange is one all-reduce over the flat buffer.
_GRAD_SLOTS = None


def set_grad_slots(table):
    global _GRAD_SLOTS
    _GRAD_SLOTS = table
    _SLOT_HANDED.clear()


_SLOT_HANDED = {}        # parameter address -> id of the backward pass (autograd graph task) that last received its slot


def grad_out(param, shape=None, dtype=torch.float32):
    """Output tensor for the gradient of ``param``: its slot of the flat buffer when one is registered (and the parameter
    is not accumulating into an existing ``.grad``), else a fresh tensor.

    A module that runs TWICE in one forward pass (the discriminator ``D`` of model_ad / model_CNN_ad, reference
    mymodel.py:210-211) asks twice during one backward pass: only the first request gets the slot -- a second kernel
    writing into the same memory would overwrite the contribution autograd still holds for the sum (found by the 2-rank
    NCCL parity test: D.0.weight was twice the PET contribution).  Autograd then adds slot + fresh tensor out of place and
    ``FlatGradReducer.finish()`` copies the sum into the slot."""
    if _GRAD_SLOTS is not None and param is not None:
        hit = _GRAD_SLOTS.get(param.data_ptr())
        if hit is not None:
            slot, owner = hit
            if owner.grad is None and (shape is None or tuple(slot.shape) == tuple(shape)) and slot.dtype == dtype:
                task = torch._C._current_graph_task_id()
                key = param.data_ptr()
                if task < 0 or _SLOT_HANDED.get(key) != task:
                    _SLOT_HANDED[key] = task
                    return slot.detach()    # a fresh alias: autograd adopts it as .grad only if nobody else holds it
    return torch.empty(tuple(param.shape) if shape is None else tuple(shape), dtype=dtype, device=param.device)


def conv_impl():
    """TMF_CONV_IMPL = auto | direct | umma  (bring-up / cross-check switch; default auto)."""
    return {"auto": L.CONV_AUTO, "direct": L.CONV_DIRECT, "umma": L.CONV_UMMA}[os.environ.get("TMF_CONV_IMPL", "auto")]


def keep_ymax():
    """TMF_KEEP_YMAX=0: max-pool layers re-read y in the backward reduction (cross-check switch; default keeps ymax)."""
    return os.environ.get("TMF_KEEP_YMAX", "1") != "0"


def _f32c(t):
    """fp32, contiguous, plain torch.Tensor (MONAI MetaTensor inputs are unwrapped)."""
    if hasattr(t, "as_tensor"):
        t = t.as_tensor()
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


# ==============================================================================================================
# sNet conv stack  (reference models/networks.py:18-61)
# ==============================================================================================================
class SNetSpec:
    """Static description of one sNet: per layer (Cin, Cout, ksize, pool)."""

    def __init__(self, dim):
        if dim < 32 or dim % 32 != 0:
            raise ValueError(f"sNet(dim={dim}): the B200 kernels work on 8-channel vectors of dim/4 channels; "
                             f"dim must be a positive multiple of 32")
        q, h = dim // 4, dim // 2
        self.layers = [(1, q, 3, L.POOL_MAX), (q, q, 3, L.POOL_NONE), (q, h, 3, L.POOL_MAX), (h, h, 3, L.POOL_NONE),
                       (h, dim, 3, L.POOL_MAX), (dim, 2 * dim, 3, L.POOL_NONE), (2 * dim, dim, 1, L.POOL_AVG)]
        self.dim = dim


class SNetSegment:
    """Layers [l0, l1) of an sNet, passed to ``SNetFunction.apply`` in the place of the spec: a segmented run (module hooks on
    the blocks, Grad-CAM; DESIGN section 3.7) chains one autograd node per segment, split at the exposed block outputs.
    A segment with l0 > 0 consumes ``src``, the bf16 NDHWC twins of its fp32 inputs (what the previous segment returned);
    a segment with l1 < 7 returns the fp32 block outputs followed by their bf16 twins (not differentiable)."""

    def __init__(self, spec, l0, l1, src=None):
        self.spec, self.l0, self.l1, self.src = spec, l0, l1, src


class ConvPack:
    """bf16 operand packs of one Conv3d weight -- wf[tap][Cout][Cin] (forward) and wd[taps-1-tap][Cin][Cout] (dgrad) -- kept
    across steps.  They are fresh while ``weight._version`` is the one they were packed from: torch in-place updates
    (``torch.optim``, ``load_state_dict``) bump it and force a repack; ``optim.FusedAdam`` rewrites the packs from its own
    kernel (the weight's version does not move), so a train step on FusedAdam has no pack launches at all."""

    def __init__(self):
        self.wf = self.wd = None
        self.version, self.ptr = None, None

    def stale(self, w):
        cout, cin, k = w.shape[0], w.shape[1], w.shape[2]
        taps = k ** 3
        if self.wf is None or self.ptr != w.data_ptr() or self.wf.device != w.device:
            self.wf = torch.empty((taps, cout, cin), dtype=torch.bfloat16, device=w.device)
            self.wd = torch.empty((taps, cin, cout), dtype=torch.bfloat16, device=w.device)
            self.version, self.ptr = None, w.data_ptr()
        if getattr(w, "_tmf_pack_cache", None) is not self:
            w._tmf_pack = (self.wf, self.wd, cout, cin, taps)      # optim.FusedAdam reads these
            w._tmf_pack_cache = self
        return self.version != w._version

    def mark(self, w):
        self.version = w._version


class EncPack:
    """bf16 hi / lo copies of one encoder's five weight matrices (the operand pack of csrc/enc_fused.cu: per matrix
    [hi | lo], in the order Wq, Wkv, Wo, W1, W2), kept across steps like ``ConvPack``: fresh while every weight's ``_version`` is
    the one it was packed from; ``optim.FusedAdam`` rewrites the hi / lo values from its own kernel (``_tmf_encpack``), so a
    train step on FusedAdam has no ``tmf_encoder_pack_weights`` launches (6 per ``model_ad`` step before)."""

    def __init__(self):
        self.pack, self.key, self.versions = None, None, {}

    def stale(self, ws, mlp):
        key = tuple(w.data_ptr() for w in ws) + (str(ws[0].device),)
        if self.pack is None or key != self.key:
            self.pack = torch.empty(int(L.load().tmf_encoder_pack_bytes(int(mlp))) // 2, dtype=torch.bfloat16, device=ws[0].device)
            self.key, self.versions = key, {}
        off = 0
        for w in ws:
            n = w.numel()
            if getattr(w, "_tmf_pack_cache", None) is not self or getattr(w, "_tmf_encpack", (None,))[0] is None \
                    or w._tmf_encpack[0].data_ptr() != self.pack.data_ptr() + 2 * off:
                w._tmf_encpack = (self.pack[off:off + n], self.pack[off + n:off + 2 * n])     # optim.FusedAdam reads these
                w._tmf_pack_cache = self
            off += 2 * n
        return any(self.versions.get(w.data_ptr()) != w._version for w in ws)

    def mark(self, w):
        self.versions[w.data_ptr()] = w._version


# Bumped whenever parameters or BatchNorm running statistics change behind torch's version counters (FusedAdam's kernel,
# train-mode forwards, CUDA-graph replays): the eval-mode BatchNorm folds below are rebuilt when it moves.
_PARAM_EPOCH = [0]


def bump_param_epoch():
    _PARAM_EPOCH[0] += 1


class EvalFold:
    """Eval-mode BatchNorm3d folded into one conv layer's operands (csrc/eval_ops.cu): w*scale as the bf16 pack (or fp32 for
    conv1.0) and b' = (b - running_mean)*scale + beta; plus the identity coefficients the LeakyReLU/pool pass then takes."""

    def __init__(self):
        self.sig = None
        self.wf = self.w32 = self.bias = self.ident = None

    def stale(self, l, tensors):
        w = tensors[0]
        sig = (_PARAM_EPOCH[0],) + tuple((t.data_ptr(), t._version) for t in tensors)
        if self.bias is None or self.bias.device != w.device:
            cout, cin, k = w.shape[0], w.shape[1], w.shape[2]
            if l == 0:
                self.w32 = torch.empty_like(w)
            else:
                self.wf = torch.empty((k ** 3, cout, cin), dtype=torch.bfloat16, device=w.device)
            self.bias = torch.empty(cout, dtype=torch.float32, device=w.device)
            self.ident = torch.zeros(4 * cout, dtype=torch.float32, device=w.device)
            self.ident[:cout] = 1.0
            self.ident[3 * cout:] = 1.0
            self.sig = None
        return sig != self.sig, sig


def refresh_eval_folds(folds, l, tensors, bn_eps):
    """Rebuild the ``EvalFold`` of layer l of one or two towers where it is stale (one ``tmf_fold_bn_pack`` launch for the
    group).  tensors[t] = (conv.weight, conv.bias, bn.weight, bn.bias, running_mean, running_var) of tower t."""
    state = [fo.stale(l, list(ts)) for fo, ts in zip(folds, tensors)]
    if any(st for st, _ in state):
        w = tensors[0][0]
        L.call("tmf_fold_bn_pack", len(folds), *[L.ptrs([ts[i] for ts in tensors]) for i in range(6)],
               L.ptrs([fo.wf for fo in folds]), L.ptrs([fo.w32 for fo in folds]), L.ptrs([fo.bias for fo in folds]),
               w.shape[0], w.shape[1], w.shape[2], float(bn_eps))
        for fo, (_, sig) in zip(folds, state):
            fo.sig = sig


class SNetRun:
    """Per-call settings of the conv stack: train / eval, whether autograd is recording (``torch.is_grad_enabled()`` at
    the call site: inside ``Function.forward`` grad mode is always off), and the hyper-parameters read from the
    ``nn.BatchNorm3d`` / ``nn.LeakyReLU`` children -- per layer (eps, momentum, negative_slope)."""

    def __init__(self, training, grad_enabled, hyper=None, packs=None, folds=None, sync_group=False, keep=None):
        self.training, self.grad_enabled = bool(training), bool(grad_enabled)
        self.hyper = hyper if hyper is not None else [(BN_EPS, BN_MOMENTUM, LRELU_SLOPE)] * 7
        self.packs = packs              # per tower: 7 ConvPack (index 0 unused: conv1.0 consumes the fp32 weight)
        self.folds = folds              # per tower: 7 EvalFold (inference path: BatchNorm folded into the conv operands)
        # False: per-rank BatchNorm statistics (DDP semantics, the default).  None / a process group: the BatchNorm3d children
        # are nn.SyncBatchNorm (torch.nn.SyncBatchNorm.convert_sync_batchnorm(model)): statistics over the GLOBAL batch
        self.sync_group = sync_group
        # per tower: a list (or None) that the folded eval path appends (input activation, y) to, layer by layer (LRP)
        self.keep = keep


def _sync_world(group):
    """World size of the SyncBatchNorm exchange (1: nothing to exchange)."""
    import torch.distributed as dist
    if group is False or not (dist.is_available() and dist.is_initialized()):
        return 1
    return dist.get_world_size(group)


def _allreduce_stat_rows(bufs, group):
    """SyncBatchNorm: replace the per-CTA partial rows of every tower's statistics buffer by the sum over all ranks (row 0 =
    the global totals, the other rows zero), so that the finalize kernels see global-batch statistics."""
    import torch.distributed as dist
    tot = torch.stack([b.sum(0) for b in bufs])
    dist.all_reduce(tot, group=group)
    for b, t in zip(bufs, tot):
        b.zero_()
        b[0].copy_(t)


def wgrad_workspace(ng, impl, B, D, H, W, cin, cout, ks, dev):
    """Caller-owned scratch for the split-K partials of the tcgen05 weight-gradient kernel (None if not needed)."""
    n = int(L.load().tmf_conv3d_wgrad_workspace_bytes(ng, impl, B, D, H, W, cin, cout, ks))
    return torch.empty(n, dtype=torch.uint8, device=dev) if n > 0 else None


def _pooled(D, H, W, pool):
    return (D, H, W) if pool == L.POOL_NONE else (D // 2, H // 2, W // 2)


class SNetFunction(torch.autograd.Function):
    """Both towers (or one) of the 3D-CNN encoder as ONE autograd node.

    apply(spec, run, buffers, ng, x_0[, x_1], *params) with run an ``SNetRun`` and params = for each tower, for each of the 7 layers:
    conv.weight, conv.bias, bn.weight, bn.bias;  buffers[t][l] = (running_mean, running_var, num_batches_tracked).
    Returns one fp32 tensor per tower with logical shape (B, dim, d, h, w) in channels-last-3d memory, i.e. the
    token matrix (B, d*h*w, dim) is a free view of it.
    """

    @staticmethod
    def forward(ctx, spec, run, buffers, ng, *args):
        training = run.training
        seg = spec if isinstance(spec, SNetSegment) else None
        if seg is not None:
            spec = seg.spec
        l0, l1 = (seg.l0, seg.l1) if seg is not None else (0, len(spec.layers))
        tap_out = l1 < len(spec.layers)
        params = args[ng:]
        assert len(params) == ng * 7 * 4
        if l0 == 0:
            xs = [_f32c(a) for a in args[:ng]]
            B, cin0, D, H, W = xs[0].shape
            if cin0 != 1:
                raise RuntimeError(f"sNet expects single-channel volumes (B,1,D,H,W); got {tuple(xs[0].shape)}")
            for x in xs:
                if tuple(x.shape) != tuple(xs[0].shape):
                    raise RuntimeError("MRI and PET volumes must have the same shape")
        else:
            xs = seg.src                                    # bf16 twins of the fp32 block outputs args[:ng]
            B, D, H, W, cin0 = xs[0].shape
            if cin0 != spec.layers[l0][0] or any(tuple(x.shape) != tuple(xs[0].shape) for x in xs):
                raise RuntimeError(f"sNet segment from layer {l0}: unexpected input {tuple(xs[0].shape)}")
        dev = xs[0].device
        need_wgrad = run.grad_enabled and any(ctx.needs_input_grad[4 + ng:])
        need_xgrad = run.grad_enabled and any(ctx.needs_input_grad[4:4 + ng])     # saliency: d / d input volume
        need_grad = need_wgrad or need_xgrad
        impl = conv_impl()
        P = lambda t, l, k: params[(t * 7 + l) * 4 + k]
        if not training and not need_grad and run.folds is not None and os.environ.get("TMF_EVAL_FOLD", "1") != "0":
            return SNetFunction._eval_forward(ctx, spec, run, buffers, ng, xs, P, impl, l0, l1)
        if training:
            bump_param_epoch()                              # running statistics are about to change
        saved = []
        act = xs
        dims = (D, H, W)
        sync_world = _sync_world(run.sync_group) if training else 1
        for l in range(l0, l1):
            cin, cout, ks, pool = spec.layers[l]
            Dl, Hl, Wl = dims
            count = B * Dl * Hl * Wl
            bn_eps, bn_momentum, slope = run.hyper[l]
            y = [torch.empty((B, Dl, Hl, Wl, cout), dtype=torch.bfloat16, device=dev) for _ in range(ng)]
            # per-CTA partial rows, summed in a fixed order by tmf_bn_finalize (deterministic; never zeroed)
            stats = L.stat_buffers(ng, cout, dev) if training else None
            w = [P(t, l, 0) for t in range(ng)]
            b = [P(t, l, 1) for t in range(ng)]
            wd = None
            if l == 0:
                L.call("tmf_conv1_fwd", ng, L.ptrs(act), L.ptrs(w), L.ptrs(b), L.ptrs(y), L.ptrs(stats),
                       B, Dl, Hl, Wl, cout, impl)
            else:
                taps = ks ** 3
                if run.packs is not None:
                    caches = [run.packs[t][l] for t in range(ng)]
                    stale = [c.stale(wt) for c, wt in zip(caches, w)]
                    wf, wd = [c.wf for c in caches], [c.wd for c in caches]
                    if any(stale):
                        L.call("tmf_pack_conv_weights", ng, L.ptrs(w), L.ptrs(wf), L.ptrs(wd), cout, cin, ks)
                        for c, wt in zip(caches, w):
                            c.mark(wt)
                else:
                    wf = [torch.empty((taps, cout, cin), dtype=torch.bfloat16, device=dev) for _ in range(ng)]
                    if need_grad:
                        wd = [torch.empty((taps, cin, cout), dtype=torch.bfloat16, device=dev) for _ in range(ng)]
                    L.call("tmf_pack_conv_weights", ng, L.ptrs(w), L.ptrs(wf), L.ptrs(wd), cout, cin, ks)
                L.call("tmf_conv3d_fwd", ng, L.ptrs(act), L.ptrs(wf), L.ptrs(b), L.ptrs(y), L.ptrs(stats),
                       B, Dl, Hl, Wl, cin, cout, ks, impl, tag=f"tmf_conv3d_fwd@L{l}")
            if training and sync_world > 1:
                _allreduce_stat_rows(stats, run.sync_group)           # SyncBatchNorm: global-batch mean / variance
                count *= sync_world
            coef = list(torch.empty((ng, 4 * cout), dtype=torch.float32, device=dev).unbind(0))
            L.call("tmf_bn_finalize", ng, L.ptrs(stats), L.ptrs([P(t, l, 2) for t in range(ng)]),
                   L.ptrs([P(t, l, 3) for t in range(ng)]), L.ptrs([buffers[t][l][0] for t in range(ng)]),
                   L.ptrs([buffers[t][l][1] for t in range(ng)]), L.ptrs([buffers[t][l][2] for t in range(ng)]),
                   L.ptrs(coef), cout, count, bn_momentum, bn_eps, int(training))
            last = l == len(spec.layers) - 1
            Do, Ho, Wo = _pooled(Dl, Hl, Wl, pool)
            out = [torch.empty((B, Do, Ho, Wo, cout), dtype=torch.float32 if last else torch.bfloat16, device=dev)
                   for _ in range(ng)]
            dual = tap_out and l == l1 - 1                  # exposed block output: fp32 value + the bf16 operand
            out32 = [torch.empty((B, Do, Ho, Wo, cout), dtype=torch.float32, device=dev) for _ in range(ng)] if dual else None
            ymax = None
            if need_grad and pool == L.POOL_MAX and keep_ymax():
                # max-pool layers keep the pre-BN value behind every window maximum: the backward reduction then reads
                # 1/8 of the voxels instead of all of y
                ymax = [torch.empty((B, Do, Ho, Wo, cout), dtype=torch.bfloat16, device=dev) for _ in range(ng)]
                if dual:
                    L.call("tmf_bn_act_pool_fwd_keepmax_dual", ng, L.ptrs(y), L.ptrs(coef), L.ptrs(out), L.ptrs(out32),
                           L.ptrs(ymax), B, Dl, Hl, Wl, cout, slope, tag=f"tmf_bn_act_pool_fwd@L{l}")
                else:
                    L.call("tmf_bn_act_pool_fwd_keepmax", ng, L.ptrs(y), L.ptrs(coef), L.ptrs(out), L.ptrs(ymax), int(last),
                           B, Dl, Hl, Wl, cout, slope, tag=f"tmf_bn_act_pool_fwd@L{l}")
            elif dual:
                L.call("tmf_bn_act_pool_fwd_dual", ng, L.ptrs(y), L.ptrs(coef), L.ptrs(out), L.ptrs(out32), B, Dl, Hl, Wl,
                       cout, pool, slope, tag=f"tmf_bn_act_pool_fwd@L{l}")
            else:
                L.call("tmf_bn_act_pool_fwd", ng, L.ptrs(y), L.ptrs(coef), L.ptrs(out), int(last), B, Dl, Hl, Wl, cout,
                       pool, slope, tag=f"tmf_bn_act_pool_fwd@L{l}")
            if need_grad:
                saved.append((act, y, coef, wd, dims, ymax))
            act = out
            dims = (Do, Ho, Wo)
        ctx.spec, ctx.training, ctx.ng, ctx.saved, ctx.B = spec, training, ng, saved, B
        ctx.hyper = run.hyper
        ctx.sync_group, ctx.sync_world = run.sync_group, sync_world
        ctx.params = params if need_grad else None          # references only (gradient slots of the flat DP buffer)
        ctx.impl = impl
        ctx.need_wgrad = need_wgrad
        ctx.x_dtypes = [a.dtype for a in args[:ng]]
        ctx.l0, ctx.l1 = l0, l1
        if tap_out:
            return SNetFunction._tap_outputs(ctx, out32, act)
        outs = tuple(o.permute(0, 4, 1, 2, 3) for o in act)      # logical (B,C,d,h,w), channels-last memory
        return outs if ng > 1 else outs[0]

    @staticmethod
    def _tap_outputs(ctx, out32, twins):
        """A segment that ends at an exposed block output: the fp32 outputs (B,C,d,h,w, channels-last memory) for autograd
        and the caller's hooks, then their bf16 twins for the next segment."""
        ctx.mark_non_differentiable(*twins)
        ctx.set_materialize_grads(False)
        return tuple(o.permute(0, 4, 1, 2, 3) for o in out32) + tuple(twins)

    @staticmethod
    def _eval_forward(ctx, spec, run, buffers, ng, xs, P, impl, l0=0, l1=7):
        """Inference (val_step, reference kfold_train_adversarial.py:144-161): no statistics, no saved activations; the
        BatchNorm of every layer is folded into the conv operands once per weight / running-statistics state."""
        B, D, H, W = (xs[0].shape[0],) + tuple(xs[0].shape[2:]) if l0 == 0 else tuple(xs[0].shape[:4])
        dev = xs[0].device
        act, dims = xs, (D, H, W)
        tap_out = l1 < len(spec.layers)
        for l in range(l0, l1):
            cin, cout, ks, pool = spec.layers[l]
            Dl, Hl, Wl = dims
            bn_eps, _, slope = run.hyper[l]
            folds = [run.folds[t][l] for t in range(ng)]
            refresh_eval_folds(folds, l, [(P(t, l, 0), P(t, l, 1), P(t, l, 2), P(t, l, 3), buffers[t][l][0], buffers[t][l][1])
                                          for t in range(ng)], bn_eps)
            y = [torch.empty((B, Dl, Hl, Wl, cout), dtype=torch.bfloat16, device=dev) for _ in range(ng)]
            for t, kept in enumerate(run.keep or ()):
                if kept is not None:
                    kept.append((act[t], y[t]))
            bias = [fo.bias for fo in folds]
            if l == 0:
                L.call("tmf_conv1_fwd", ng, L.ptrs(act), L.ptrs([fo.w32 for fo in folds]), L.ptrs(bias), L.ptrs(y), L.ptrs(None),
                       B, Dl, Hl, Wl, cout, impl)
            else:
                L.call("tmf_conv3d_fwd", ng, L.ptrs(act), L.ptrs([fo.wf for fo in folds]), L.ptrs(bias), L.ptrs(y), L.ptrs(None),
                       B, Dl, Hl, Wl, cin, cout, ks, impl, tag=f"tmf_conv3d_fwd@L{l}")
            last = l == len(spec.layers) - 1
            Do, Ho, Wo = _pooled(Dl, Hl, Wl, pool)
            out = [torch.empty((B, Do, Ho, Wo, cout), dtype=torch.float32 if last else torch.bfloat16, device=dev)
                   for _ in range(ng)]
            if tap_out and l == l1 - 1:
                out32 = [torch.empty((B, Do, Ho, Wo, cout), dtype=torch.float32, device=dev) for _ in range(ng)]
                L.call("tmf_bn_act_pool_fwd_dual", ng, L.ptrs(y), L.ptrs([fo.ident for fo in folds]), L.ptrs(out),
                       L.ptrs(out32), B, Dl, Hl, Wl, cout, pool, slope, tag=f"tmf_bn_act_pool_fwd@L{l}")
                ctx.saved = None
                return SNetFunction._tap_outputs(ctx, out32, out)
            L.call("tmf_bn_act_pool_fwd", ng, L.ptrs(y), L.ptrs([fo.ident for fo in folds]), L.ptrs(out), int(last), B, Dl, Hl,
                   Wl, cout, pool, slope, tag=f"tmf_bn_act_pool_fwd@L{l}")
            act, dims = out, (Do, Ho, Wo)
        ctx.saved = None
        outs = tuple(o.permute(0, 4, 1, 2, 3) for o in act)
        return outs if ng > 1 else outs[0]

    @staticmethod
    def backward(ctx, *grads):
        spec, ng, B, training = ctx.spec, ctx.ng, ctx.B, ctx.training
        l0, l1 = ctx.l0, ctx.l1
        saved = ctx.saved
        if saved is None or len(saved) != l1 - l0:
            raise RuntimeError("sNet backward: the saved activations are gone -- backward through this forward ran "
                               "already (they are freed layer by layer; retain_graph / double backward are not "
                               "supported), or the forward ran without autograd recording")
        dev = saved[0][1][0].device
        dout = []
        for t in range(ng):
            g = grads[t]
            cout = spec.layers[l1 - 1][1]
            if g is None:
                Dl, Hl, Wl = _pooled(*saved[-1][4], spec.layers[l1 - 1][3])
                g = torch.zeros((B, Dl, Hl, Wl, cout), dtype=torch.float32, device=dev)
            else:
                g = _f32c(g.permute(0, 2, 3, 4, 1))
            dout.append(g)
        dout_fp32 = 1
        pgrads = [None] * (ng * 7 * 4)
        need_w = ctx.need_wgrad
        # frozen weights (saliency): no weight-gradient launches, no parameter .grad; BatchNorm's parameter gradients
        # still come out of tmf_bn_bwd_finalize (next to bcoef, which the input gradient needs) into scratch
        xg = [t for t in range(ng) if ctx.needs_input_grad[4 + t]]
        dxs = [None] * ng
        for l in range(l1 - 1, l0 - 1, -1):
            cin, cout, ks, pool = spec.layers[l]
            act, y, coef, wd, (Dl, Hl, Wl), ymax = saved[l - l0]
            count = B * Dl * Hl * Wl
            slope = ctx.hyper[l][2]
            if l == 0 and dout_fp32:
                # a segment of block 1 alone: its fused backward kernels read a bf16 pooled gradient
                d16 = [torch.empty(d.shape, dtype=torch.bfloat16, device=dev) for d in dout]
                L.call("tmf_narrow_f32", ng, L.ptrs(dout), L.ptrs(d16), dout[0].numel())
                dout, dout_fp32 = d16, 0
            sums = L.stat_buffers(ng, cout, dev)
            if ymax is not None:
                L.call("tmf_bn_maxpool_bwd_reduce_kept", ng, L.ptrs(dout), dout_fp32, L.ptrs(ymax), L.ptrs(coef),
                       L.ptrs(sums), B, Dl // 2, Hl // 2, Wl // 2, cout, slope,
                       tag=f"tmf_bn_act_pool_bwd_reduce@L{l}")
            else:
                L.call("tmf_bn_act_pool_bwd_reduce", ng, L.ptrs(dout), dout_fp32, L.ptrs(y), L.ptrs(coef), L.ptrs(sums),
                       B, Dl, Hl, Wl, cout, pool, slope, tag=f"tmf_bn_act_pool_bwd_reduce@L{l}")
            PG = lambda t, k: ctx.params[(t * 7 + l) * 4 + k]
            if need_w:
                dbias = [grad_out(PG(t, 1)) for t in range(ng)]
                dgamma = [grad_out(PG(t, 2)) for t in range(ng)]
                dbeta = [grad_out(PG(t, 3)) for t in range(ng)]
            else:
                dbias, dgamma, dbeta = (list(s.unbind(0)) for s in torch.empty((3, ng, cout), dtype=torch.float32, device=dev))
            bcoef = list(torch.empty((ng, 2 * cout), dtype=torch.float32, device=dev).unbind(0))
            L.call("tmf_bn_bwd_finalize", ng, L.ptrs(sums), L.ptrs(coef), L.ptrs(dgamma), L.ptrs(dbeta),
                   L.ptrs(dbias), L.ptrs(bcoef), cout, count, int(training))
            if training and ctx.sync_world > 1:
                # SyncBatchNorm: the parameter gradients above are this rank's own (the gradient exchange averages them);
                # the input gradient needs the GLOBAL means of dz and dz * xhat
                _allreduce_stat_rows(sums, ctx.sync_group)
                scratch_g = list(torch.empty((3 * ng, cout), dtype=torch.float32, device=dev).unbind(0))
                L.call("tmf_bn_bwd_finalize", ng, L.ptrs(sums), L.ptrs(coef), L.ptrs(scratch_g[:ng]), L.ptrs(scratch_g[ng:2 * ng]),
                       L.ptrs(scratch_g[2 * ng:]), L.ptrs(bcoef), cout, count * ctx.sync_world, int(training))
            if l == 0 and xg:
                if dout_fp32:
                    raise RuntimeError("sNet backward: the input gradient needs a bf16 pooled gradient into block 1")
                w0 = [PG(t, 0) for t in xg]
                dx = [torch.empty((B, 1, Dl, Hl, Wl), dtype=torch.float32, device=dev) for _ in xg]
                nws = int(L.load().tmf_conv1_dgrad_fused_workspace_bytes(len(xg), ctx.impl, B, Dl, Hl, Wl, cout))
                ws = torch.empty(nws, dtype=torch.uint8, device=dev) if nws > 0 else None
                L.call("tmf_conv1_dgrad_fused", len(xg), L.ptrs([dout[t] for t in xg]), L.ptrs([y[t] for t in xg]),
                       L.ptrs([coef[t] for t in xg]), L.ptrs([bcoef[t] for t in xg]), L.ptrs(w0), L.ptrs(dx),
                       B, Dl, Hl, Wl, cout, slope, ctx.impl, L.ptr(ws), nws)
                for t, d in zip(xg, dx):
                    dxs[t] = d if ctx.x_dtypes[t] == torch.float32 else d.to(ctx.x_dtypes[t])
            if l == 0 and not need_w:
                saved[l - l0] = None
                continue
            dw = [grad_out(PG(t, 0)) for t in range(ng)] if need_w else None
            fused_ws = 0
            if l == 0 and pool == L.POOL_MAX and not dout_fp32 and ctx.impl != L.CONV_DIRECT:
                fused_ws = int(L.load().tmf_conv1_bwd_fused_workspace_bytes(ng, B, Dl, Hl, Wl, cout))
            if fused_ws > 0:
                # block 1: BN/LeakyReLU/MaxPool backward "apply" + conv1.0 weight gradient in one pass; dy stays on chip
                ws = torch.empty(fused_ws, dtype=torch.uint8, device=dev)
                L.call("tmf_conv1_bwd_fused", ng, L.ptrs(dout), L.ptrs(y), L.ptrs(coef), L.ptrs(bcoef), L.ptrs(act),
                       L.ptrs(dw), B, Dl, Hl, Wl, cout, slope, L.ptr(ws), fused_ws)
                SNetFunction._layer_grads(ctx, pgrads, l, dw, dbias, dgamma, dbeta)
                saved[l - l0] = None
                continue
            dy = [torch.empty((B, Dl, Hl, Wl, cout), dtype=torch.bfloat16, device=dev) for _ in range(ng)]
            L.call("tmf_bn_act_pool_bwd_apply", ng, L.ptrs(dout), dout_fp32, L.ptrs(y), L.ptrs(coef), L.ptrs(bcoef),
                   L.ptrs(dy), B, Dl, Hl, Wl, cout, pool, slope, tag=f"tmf_bn_act_pool_bwd_apply@L{l}")
            if l == 0:
                nws = int(L.load().tmf_conv1_wgrad_workspace_bytes(ng, ctx.impl, Wl, cout))
                ws = torch.empty(nws, dtype=torch.uint8, device=dev) if nws > 0 else None
                L.call("tmf_conv1_wgrad", ng, L.ptrs(dy), L.ptrs(act), L.ptrs(dw), B, Dl, Hl, Wl, cout, ctx.impl,
                       L.ptr(ws), nws)
            else:
                if need_w:
                    ws = wgrad_workspace(ng, ctx.impl, B, Dl, Hl, Wl, cin, cout, ks, dev)
                    L.call("tmf_conv3d_wgrad", ng, L.ptrs(dy), L.ptrs(act), L.ptrs(dw), B, Dl, Hl, Wl, cin, cout, ks,
                           ctx.impl, L.ptr(ws), 0 if ws is None else ws.numel(), tag=f"tmf_conv3d_wgrad@L{l}")
                if l > l0 or xg:                            # a segment's first layer: only for an input that wants it
                    da = [torch.empty((B, Dl, Hl, Wl, cin), dtype=torch.bfloat16, device=dev) for _ in range(ng)]
                    L.call("tmf_conv3d_fwd", ng, L.ptrs(dy), L.ptrs(wd), L.ptrs(None), L.ptrs(da), L.ptrs(None),
                           B, Dl, Hl, Wl, cout, cin, ks, ctx.impl, tag=f"tmf_conv3d_dgrad@L{l}")
                    dout, dout_fp32 = da, 0
                if l == l0 and xg:
                    # gradient with respect to the exposed fp32 block output: the bf16 dgrad output, widened
                    da32 = [torch.empty(d.shape, dtype=torch.float32, device=dev) for d in da]
                    L.call("tmf_widen_bf16", ng, L.ptrs(da), L.ptrs(da32), da[0].numel())
                    for t in xg:
                        dxs[t] = da32[t].permute(0, 4, 1, 2, 3)
            if need_w:
                SNetFunction._layer_grads(ctx, pgrads, l, dw, dbias, dgamma, dbeta)
            saved[l - l0] = None
        ctx.saved = None
        ctx.params = None
        return (None, None, None, None) + tuple(dxs) + tuple(pgrads)

    @staticmethod
    def _layer_grads(ctx, pgrads, l, dw, dbias, dgamma, dbeta):
        for t in range(ctx.ng):
            base = (t * 7 + l) * 4
            pgrads[base + 0], pgrads[base + 1], pgrads[base + 2], pgrads[base + 3] = dw[t], dbias[t], dgamma[t], dbeta[t]


# ==============================================================================================================
# Linear / LayerNorm / attention / pooling / GRL
# ==============================================================================================================
class LinearFunction(torch.autograd.Function):
    """y = act(x W^T + b) + residual   (nn.Linear; act = exact GELU when gelu=True)."""

    @staticmethod
    def forward(ctx, x, w, b, residual, gelu):
        x2 = _f32c(x).reshape(-1, x.shape[-1])
        M, K = x2.shape
        N = w.shape[0]
        w = _f32c(w)
        y = torch.empty((M, N), dtype=torch.float32, device=x2.device)
        pre = torch.empty_like(y) if gelu else None
        res2 = _f32c(residual).reshape(M, N) if residual is not None else None
        L.call("tmf_linear_fwd", L.ptr(x2), L.ptr(w), L.ptr(None if b is None else _f32c(b)), L.ptr(res2), L.ptr(y),
               L.ptr(pre), M, K, N, int(gelu))
        ctx.save_for_backward(x2, w, pre)
        ctx.bias_ref = b                                     # reference only: its gradient slot (flat DP buffer)
        ctx.has_bias, ctx.has_res, ctx.gelu = b is not None, residual is not None, gelu
        ctx.xshape = x.shape
        return y.reshape(*x.shape[:-1], N)

    @staticmethod
    def backward(ctx, dy):
        x2, w, pre = ctx.saved_tensors
        M, K = x2.shape
        N = w.shape[0]
        dy2 = _f32c(dy).reshape(M, N)
        dres = dy2.reshape(dy.shape) if ctx.has_res else None
        if ctx.gelu:
            dpre = torch.empty_like(dy2)
            L.call("tmf_gelu_bwd", L.ptr(dy2), L.ptr(pre), L.ptr(dpre), M * N)
            dy2 = dpre
        dx = dw = db = None
        if ctx.needs_input_grad[0]:
            dx = torch.empty((M, K), dtype=torch.float32, device=dy2.device)
            L.call("tmf_linear_dgrad", L.ptr(dy2), L.ptr(w), L.ptr(dx), M, K, N, 0)
            dx = dx.reshape(ctx.xshape)
        if ctx.needs_input_grad[1] or (ctx.has_bias and ctx.needs_input_grad[2]):
            dw = grad_out(w, (N, K))
            db = grad_out(ctx.bias_ref, (N,)) if ctx.has_bias else None
            ws, nws = L.scratch(dy2.device)
            L.call("tmf_linear_wgrad", L.ptr(dy2), L.ptr(x2), L.ptr(dw), L.ptr(db), M, K, N, L.ptr(ws), nws)
        return dx, dw, db, dres, None


def linear(x, w, b=None, residual=None, gelu=False):
    return LinearFunction.apply(x, w, b, residual, gelu)


class LayerNormFunction(torch.autograd.Function):
    """y = LayerNorm(x) * gamma + beta (+ residual)."""

    @staticmethod
    def forward(ctx, x, gamma, beta, residual, eps):
        x2 = _f32c(x).reshape(-1, x.shape[-1])
        rows, dim = x2.shape
        y = torch.empty_like(x2)
        mean = torch.empty(rows, dtype=torch.float32, device=x2.device)
        rstd = torch.empty_like(mean)
        res2 = _f32c(residual).reshape(rows, dim) if residual is not None else None
        g = _f32c(gamma)
        L.call("tmf_layernorm_fwd", L.ptr(x2), L.ptr(g), L.ptr(_f32c(beta)), L.ptr(res2), L.ptr(y), L.ptr(mean),
               L.ptr(rstd), rows, dim, eps)
        ctx.save_for_backward(x2, g, mean, rstd)
        ctx.beta_ref = beta
        ctx.has_res = residual is not None
        return y.reshape(x.shape)

    @staticmethod
    def backward(ctx, dy):
        x2, g, mean, rstd = ctx.saved_tensors
        rows, dim = x2.shape
        dy2 = _f32c(dy).reshape(rows, dim)
        dx = torch.empty_like(x2)
        dgamma, dbeta = grad_out(g, (dim,)), grad_out(ctx.beta_ref, (dim,))
        ws, nws = L.scratch(x2.device)
        L.call("tmf_layernorm_bwd", L.ptr(dy2), L.ptr(x2), L.ptr(g), L.ptr(mean), L.ptr(rstd), L.ptr(dx), L.ptr(dgamma),
               L.ptr(dbeta), rows, dim, 0, L.ptr(ws), nws)
        return dx.reshape(dy.shape), dgamma, dbeta, (dy if ctx.has_res else None), None


def layer_norm(x, gamma, beta, residual=None, eps=LN_EPS):
    return LayerNormFunction.apply(x, gamma, beta, residual, eps)


class AttentionCoreFunction(torch.autograd.Function):
    """softmax(q k^T * scale) v per head on short token sequences; q (B,Nq,h*dh), kv (B,Nk,2*h*dh).  With an ``AttnTap``
    it also returns the reference's ``dots`` and ``attn`` (DESIGN section 3.8)."""

    @staticmethod
    def forward(ctx, q, kv, heads, scale, tap=None):
        q, kv = _f32c(q), _f32c(kv)
        B, Nq, inner = q.shape
        Nk = kv.shape[1]
        dh = inner // heads
        out = torch.empty_like(q)
        lse = torch.empty((B, heads, Nq), dtype=torch.float32, device=q.device)
        L.call("tmf_attn_fwd", L.ptr(q), L.ptr(kv), L.ptr(out), L.ptr(lse), B, Nq, Nk, heads, dh, float(scale))
        ctx.save_for_backward(q, kv, out, lse)
        ctx.heads, ctx.scale = heads, float(scale)
        ctx.tap = tap
        if tap is None:
            return out
        dots, attn = attn_scores(q, kv, heads, scale, lse)
        tap.arm(kv, heads, None)
        ctx.mark_non_differentiable(dots)
        ctx.set_materialize_grads(False)
        return out, dots, attn

    @staticmethod
    def backward(ctx, dout, ddots=None, dattn=None):
        q, kv, out, lse = ctx.saved_tensors
        B, Nq, inner = q.shape
        Nk = kv.shape[1]
        if ctx.tap is not None:
            ctx.tap.check(dattn)
        dq, dkv = torch.empty_like(q), torch.empty_like(kv)
        if dout is None:
            dout = torch.zeros_like(out)
        L.call("tmf_attn_bwd", L.ptr(_f32c(dout)), L.ptr(q), L.ptr(kv), L.ptr(out), L.ptr(lse), L.ptr(dq), L.ptr(dkv),
               B, Nq, Nk, ctx.heads, inner // ctx.heads, ctx.scale)
        return dq, dkv, None, None, None


def attention_core(q, kv, heads, scale, tap=None):
    return AttentionCoreFunction.apply(q, kv, heads, scale, tap)


# ==============================================================================================================
# Attention probabilities for module hooks and attention maps   (csrc/attention_mma.cu, DESIGN section 3.8)
# ==============================================================================================================
def attn_scores(q, kv, heads, scale, lse):
    """(dots, attn), fp32 (B, heads, Nq, Nk): scale * q_h k_h^T and exp(dots - lse), with the attention core's operands."""
    B, Nq, inner = q.shape
    Nk = kv.shape[1]
    dots = torch.empty((B, heads, Nq, Nk), dtype=torch.float32, device=q.device)
    attn = torch.empty_like(dots)
    L.call("tmf_attn_scores", 0, L.ptr(q), L.ptr(kv), L.ptr(lse), L.ptr(dots), L.ptr(attn), B, Nq, Nk, heads, inner // heads,
           float(scale))
    return dots, attn


def attn_scores_grad(dout, kv, heads):
    """dL/d attn = dO_h v_h^T, fp32 (B, heads, Nq, Nk), from dL/d out (B, Nq, heads*dh)."""
    dout = _f32c(dout)
    B, Nq, inner = dout.shape
    Nk = kv.shape[1]
    dattn = torch.empty((B, heads, Nq, Nk), dtype=torch.float32, device=dout.device)
    L.call("tmf_attn_scores", 1, L.ptr(dout), L.ptr(kv), L.ptr(None), L.ptr(dattn), L.ptr(None), B, Nq, Nk, heads,
           inner // heads, 1.0)
    return dattn


def attn_relevance(attn, dattn=None, r=None, accumulate=False):
    """Head-averaged map M = mean_h attn (or mean_h max(attn * dattn, 0)), (B, Nq, Nk), and the key relevance
    r = mean_i M, (B, Nk), written into ``r`` when given (added to it with ``accumulate``).  Returns (M, r)."""
    attn = _f32c(attn.detach())
    B, heads, Nq, Nk = attn.shape
    if dattn is not None:
        dattn = _f32c(dattn.detach())
        if dattn.shape != attn.shape:
            raise ValueError("attn_relevance: attn and dattn must have the same shape")
    M = torch.empty((B, Nq, Nk), dtype=torch.float32, device=attn.device)
    acc = r is not None and accumulate
    if r is None:
        r = torch.empty((B, Nk), dtype=torch.float32, device=attn.device)
    elif tuple(r.shape) != (B, Nk) or r.dtype != torch.float32 or not r.is_contiguous():
        raise ValueError(f"attn_relevance: r must be a contiguous fp32 ({B}, {Nk}) tensor")
    L.call("tmf_attn_relevance", L.ptr(attn), L.ptr(dattn), L.ptr(M), L.ptr(r), B, heads, Nq, Nk, int(acc))
    return M, r


def map_resample(lo, size, normalize=True):
    """``lo``: fp32 (ng, B, d, h, w) maps -> ng fp32 (B, 1, D, H, W) maps, trilinear (align_corners=False) to ``size``
    and normalised per sample to [0, 1] when ``normalize``: Grad-CAM's resampling pass (csrc/gradcam.cu)."""
    lo = _f32c(lo)
    ng, B, d, h, w = lo.shape
    D, H, W = (int(s) for s in size)
    outs = [torch.empty((B, 1, D, H, W), dtype=torch.float32, device=lo.device) for _ in range(ng)]
    for i in range(0, ng, 2):
        n = min(2, ng - i)
        nws = int(L.load().tmf_map_resample_workspace_bytes(n, B, d, h, w, D, H, W, int(normalize)))
        if nws < 0:
            raise ValueError(f"map_resample: unsupported problem B={B} {d}x{h}x{w} -> {D}x{H}x{W}")
        ws = torch.empty(max(nws, 1), dtype=torch.uint8, device=lo.device)
        L.call("tmf_map_resample", n, L.ptr(lo[i:i + n]), L.ptrs(outs[i:i + n]), B, d, h, w, D, H, W, int(normalize),
               L.ptr(ws), nws)
    return outs


class AttnTap:
    """What ties an attention node that exposes ``attn`` to the ``AttnTapFunction`` node behind its output.  The tap node's
    backward turns the gradient of the output into dL/d attn (``tmf_attn_scores`` mode 1) and hands it to autograd; the
    attention node's backward then checks that the gradient it receives for ``attn`` is that very tensor, unmodified --
    the probabilities may only be observed, never feed anything else."""

    def __init__(self):
        self.kv = self.heads = self.chain = None
        self.dattn, self.version = None, None
        self.stash = None

    def arm(self, kv, heads, chain):
        """``chain(dy) -> (dO, stash)``: the gradient of the attention output from that of the node's output (fused encoder:
        its chain backward, whose results ``stash`` the encoder's backward reuses; attention core: the identity)."""
        self.kv, self.heads, self.chain = kv, heads, chain

    def grad(self, dy):
        dout, self.stash = self.chain(dy) if self.chain is not None else (dy, None)
        self.dattn = attn_scores_grad(dout, self.kv, self.heads)
        self.version = self.dattn._version
        self.kv = self.chain = None
        return self.dattn

    def check(self, dattn):
        if dattn is not None and (dattn is not self.dattn or dattn._version != self.version):
            # this backward pass ends here: join the weight-gradient work that encoders behind this one already put on the
            # side stream (the engine callback that would have joined it is dropped with the pass)
            join_side_streams()
            raise NotImplementedError("attention probabilities may only be observed: a gradient other than the one the "
                                      "model's own output gives reached `attn` (a tensor hook on it returned or modified a "
                                      "gradient, or `attn` entered a loss). Clone `attn` to compute with it")
        self.dattn = None


class AttnTapFunction(torch.autograd.Function):
    """Identity on an attention node's output ``y`` that also consumes its ``attn``: backward returns dy unchanged and
    dL/d attn as ``attn``'s gradient, so that tensor hooks on ``attn`` see it."""

    @staticmethod
    def forward(ctx, y, attn, tap):
        ctx.tap = tap
        return y.view_as(y)

    @staticmethod
    def backward(ctx, dy):
        return dy, ctx.tap.grad(dy), None


def attn_tap(y, attn, tap):
    if not (torch.is_grad_enabled() and attn.requires_grad):
        return y
    return AttnTapFunction.apply(y, attn, tap)


# Side stream for work that is off the backward pass's critical path (the encoders' weight gradients): launched there, it
# overlaps the next encoder's dgrad chain; the launching stream waits for it when autograd finishes the backward pass
# (engine callback), i.e. before anything can consume the gradients.  Under CUDA-graph capture this becomes a parallel branch.
_SIDE = {}
_SIDE_PENDING = []


def _side_stream(device):
    key = (device.index, torch.cuda.current_stream(device).cuda_stream)
    st = _SIDE.get(key)
    if st is None:
        st = torch.cuda.Stream(device=device)
        _SIDE[key] = st
    return st


def join_side_streams():
    """Make the current stream wait for everything launched on the side stream (idempotent)."""
    while _SIDE_PENDING:
        torch.cuda.current_stream().wait_event(_SIDE_PENDING.pop())


class EncoderFunction(torch.autograd.Function):
    """One ``Transformer(depth=1)`` encoder (reference models/networks.py:215-230) with cross-attention context, as three
    forward and five backward launches (csrc/enc_fused.cu + the attention core):
        a = Attn(LN1(x), ctx) + x;   y = LNf(FF(LN2(a)) + a) (+ x when ``add_input``: the caller's outer residual).
    params = (ln1_w, ln1_b, wq, wkv, wo, bo, ln2_w, ln2_b, w1, b1, w2, b2, lnf_w, lnf_b)."""

    @staticmethod
    def forward(ctx, x, context, heads, scale, add_input, eps1, eps2, epsf, pack_cache, tap, *params):
        ln1_w, ln1_b, wq, wkv, wo, bo, ln2_w, ln2_b, w1, b1, w2, b2, lnf_w, lnf_b = [_f32c(t) for t in params]
        x3, c3 = _f32c(x), _f32c(context)
        B, Nq, dim = x3.shape
        Nk = c3.shape[1]
        Mx, Mc, mlp = B * Nq, B * Nk, w1.shape[0]
        dev = x3.device
        E = lambda *shape: torch.empty(shape, dtype=torch.float32, device=dev)
        h1, mean1, rstd1, q, kv = E(Mx, dim), E(Mx), E(Mx), E(B, Nq, dim), E(B, Nk, 2 * dim)
        # bf16 hi / lo copies of the five weight matrices for the split-weight GEMMs (one launch; the backward pass reuses
        # them).  TMF_ENC_BF16=0: three-pass TF32 straight from the fp32 weights (pack = NULL).
        pack = None
        if os.environ.get("TMF_ENC_BF16", "1") != "0":
            ws5 = (wq, wkv, wo, w1, w2)
            cached = pack_cache is not None and all(w is t for w, t in zip(ws5, (params[2], params[3], params[4], params[8], params[10])))
            if cached:                                      # the module's pack, refreshed by FusedAdam between steps
                if pack_cache.stale(ws5, mlp):
                    L.call("tmf_encoder_pack_weights", L.ptr(wq), L.ptr(wkv), L.ptr(wo), L.ptr(w1), L.ptr(w2), mlp, L.ptr(pack_cache.pack))
                    for w in ws5:
                        pack_cache.mark(w)
                pack = pack_cache.pack
            else:
                pack = torch.empty(int(L.load().tmf_encoder_pack_bytes(int(mlp))) // 2, dtype=torch.bfloat16, device=dev)
                L.call("tmf_encoder_pack_weights", L.ptr(wq), L.ptr(wkv), L.ptr(wo), L.ptr(w1), L.ptr(w2), mlp, L.ptr(pack))
        L.call("tmf_encoder_proj_fwd", L.ptr(x3), L.ptr(c3), L.ptr(ln1_w), L.ptr(ln1_b), L.ptr(wq), L.ptr(wkv), L.ptr(h1),
               L.ptr(mean1), L.ptr(rstd1), L.ptr(q), L.ptr(kv), Mx, Mc, float(eps1), L.ptr(pack))
        o, lse = E(B, Nq, dim), E(B, heads, Nq)
        L.call("tmf_attn_fwd", L.ptr(q), L.ptr(kv), L.ptr(o), L.ptr(lse), B, Nq, Nk, heads, dim // heads, float(scale))
        a, h2, mean2, rstd2, pre, f, g = E(Mx, dim), E(Mx, dim), E(Mx), E(Mx), E(Mx, mlp), E(Mx, mlp), E(Mx, dim)
        meanf, rstdf, y = E(Mx), E(Mx), E(B, Nq, dim)
        L.call("tmf_encoder_chain_fwd", L.ptr(o), L.ptr(x3), L.ptr(wo), L.ptr(bo), L.ptr(ln2_w), L.ptr(ln2_b), L.ptr(w1),
               L.ptr(b1), L.ptr(w2), L.ptr(b2), L.ptr(lnf_w), L.ptr(lnf_b), L.ptr(a), L.ptr(h2), L.ptr(mean2), L.ptr(rstd2),
               L.ptr(pre), L.ptr(f), L.ptr(g), L.ptr(meanf), L.ptr(rstdf), L.ptr(y), Mx, mlp, int(add_input), float(eps2),
               float(epsf), L.ptr(pack))
        ctx.save_for_backward(x3, c3, h1, mean1, rstd1, q, kv, o, lse, a, h2, mean2, rstd2, pre, f, g, meanf, rstdf,
                              ln1_w, wq, wkv, wo, ln2_w, w1, w2, lnf_w)
        ctx.pack = pack
        ctx.param_refs = params                              # references only: gradient slots of the flat DP buffer
        ctx.cfg = (heads, float(scale), bool(add_input), B, Nq, Nk, dim, mlp)
        ctx.tap = tap
        if tap is None:
            return y.reshape(x.shape)
        # attention maps (DESIGN section 3.8): the probabilities behind o, one more launch
        dots, attn = attn_scores(q, kv, heads, scale, lse)
        chain_in = (g, a, pre, wo, w1, w2, ln2_w, lnf_w, mean2, rstd2, meanf, rstdf)
        cfg = ctx.cfg
        tap.arm(kv, heads, lambda dy: EncoderFunction._chain_bwd(cfg, params, pack, chain_in, dy))
        ctx.mark_non_differentiable(dots)
        ctx.set_materialize_grads(False)
        return y.reshape(x.shape), dots, attn

    @staticmethod
    def _chain_bwd(cfg, P, pack, saved, dy):
        """tmf_encoder_chain_bwd: the gradients of the attention output (dout), of the residual input (dxp) and of the rows
        behind them, plus the gradients of the two LayerNorms it covers."""
        g, a, pre, wo, w1, w2, ln2_w, lnf_w, mean2, rstd2, meanf, rstdf = saved
        heads, scale, add_input, B, Nq, Nk, dim, mlp = cfg
        Mx = B * Nq
        dev = g.device
        E = lambda *shape: torch.empty(shape, dtype=torch.float32, device=dev)
        d_ln2_w, d_ln2_b, d_lnf_w, d_lnf_b = grad_out(P[6]), grad_out(P[7]), grad_out(P[12]), grad_out(P[13])
        ws, nws = L.scratch(dev)
        dy2 = _f32c(dy).reshape(Mx, dim)
        dg, dp, da, dout, dxp = E(Mx, dim), E(Mx, mlp), E(Mx, dim), E(B, Nq, dim), E(Mx, dim)
        L.call("tmf_encoder_chain_bwd", L.ptr(dy2), L.ptr(g), L.ptr(a), L.ptr(pre), L.ptr(wo), L.ptr(w1), L.ptr(w2), L.ptr(ln2_w),
               L.ptr(lnf_w), L.ptr(mean2), L.ptr(rstd2), L.ptr(meanf), L.ptr(rstdf), L.ptr(dg), L.ptr(dp), L.ptr(da),
               L.ptr(dout), L.ptr(dxp), L.ptr(d_lnf_w), L.ptr(d_lnf_b), L.ptr(d_ln2_w), L.ptr(d_ln2_b), Mx, mlp,
               int(add_input), L.ptr(pack), L.ptr(ws), nws)
        return dout, (dy, dg, dp, da, dout, dxp, d_ln2_w, d_ln2_b, d_lnf_w, d_lnf_b)

    @staticmethod
    def backward(ctx, dy, ddots=None, dattn=None):
        (x3, c3, h1, mean1, rstd1, q, kv, o, lse, a, h2, mean2, rstd2, pre, f, g, meanf, rstdf,
         ln1_w, wq, wkv, wo, ln2_w, w1, w2, lnf_w) = ctx.saved_tensors
        heads, scale, add_input, B, Nq, Nk, dim, mlp = ctx.cfg
        Mx, Mc = B * Nq, B * Nk
        dev = x3.device
        E = lambda *shape: torch.empty(shape, dtype=torch.float32, device=dev)
        P = ctx.param_refs
        G = lambda i: grad_out(P[i])
        stash = None
        if ctx.tap is not None:
            ctx.tap.check(dattn)
            stash, ctx.tap.stash = ctx.tap.stash, None
            if dy is None:
                dy = torch.zeros((B, Nq, dim), dtype=torch.float32, device=dev)
        if stash is not None and stash[0] is dy:
            # the tap node ran the chain backward on this very gradient to get dL/d attn: its results are reused
            _, dg, dp, da, dout, dxp, d_ln2_w, d_ln2_b, d_lnf_w, d_lnf_b = stash
            d_ln1_w, d_ln1_b, d_wq, d_wkv, d_wo, d_bo = [G(i) for i in range(6)]
            d_w1, d_b1, d_w2, d_b2 = [G(i) for i in range(8, 12)]
            ws, nws = L.scratch(dev)
        else:
            d_ln1_w, d_ln1_b, d_wq, d_wkv, d_wo, d_bo, d_ln2_w, d_ln2_b, d_w1, d_b1, d_w2, d_b2, d_lnf_w, d_lnf_b = [G(i) for i in range(14)]
            ws, nws = L.scratch(dev)
            dy2 = _f32c(dy).reshape(Mx, dim)
            dg, dp, da, dout, dxp = E(Mx, dim), E(Mx, mlp), E(Mx, dim), E(B, Nq, dim), E(Mx, dim)
            L.call("tmf_encoder_chain_bwd", L.ptr(dy2), L.ptr(g), L.ptr(a), L.ptr(pre), L.ptr(wo), L.ptr(w1), L.ptr(w2), L.ptr(ln2_w),
                   L.ptr(lnf_w), L.ptr(mean2), L.ptr(rstd2), L.ptr(meanf), L.ptr(rstdf), L.ptr(dg), L.ptr(dp), L.ptr(da),
                   L.ptr(dout), L.ptr(dxp), L.ptr(d_lnf_w), L.ptr(d_lnf_b), L.ptr(d_ln2_w), L.ptr(d_ln2_b), Mx, mlp,
                   int(add_input), L.ptr(ctx.pack), L.ptr(ws), nws)
        dq, dkv = E(B, Nq, dim), E(B, Nk, 2 * dim)
        L.call("tmf_attn_bwd", L.ptr(dout), L.ptr(q), L.ptr(kv), L.ptr(o), L.ptr(lse), L.ptr(dq), L.ptr(dkv), B, Nq, Nk, heads,
               dim // heads, scale)
        dx, dctx = E(B, Nq, dim), E(B, Nk, dim)
        L.call("tmf_encoder_proj_bwd", L.ptr(dq), L.ptr(dkv), L.ptr(dxp), L.ptr(x3), L.ptr(ln1_w), L.ptr(mean1), L.ptr(rstd1),
               L.ptr(wq), L.ptr(wkv), L.ptr(dx), L.ptr(dctx), L.ptr(d_ln1_w), L.ptr(d_ln1_b), Mx, Mc, L.ptr(ctx.pack),
               L.ptr(ws), nws)
        if not any(ctx.needs_input_grad[10:]):
            # frozen weights (saliency, Grad-CAM): no weight-gradient launch; the LayerNorm parameter gradients above come
            # out of the input-gradient kernels anyway
            return (dx.reshape(x3.shape), dctx.reshape(c3.shape)) + (None,) * 22
        table = (ctypes_ptr_array([dq, h1, d_wq, dkv, c3, d_wkv, da, o, d_wo, d_bo, dp, h2, d_w1, d_b1, dg]))
        # all five weight gradients feed nothing downstream in this backward pass: off the critical path
        cur = torch.cuda.current_stream(dev)
        side = _side_stream(dev)
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            ws2, nws2 = L.scratch(dev)                       # the side stream's own scratch buffer
            L.call("tmf_encoder_wgrad", table, L.ptr(f), L.ptr(d_w2), L.ptr(d_b2), Mx, Mc, mlp, L.ptr(ws2), nws2)
            ev = torch.cuda.Event()
            ev.record(side)
        for t in (dq, h1, dkv, c3, da, o, dp, h2, dg, f, d_wq, d_wkv, d_wo, d_bo, d_w1, d_b1, d_w2, d_b2):
            t.record_stream(side)
        if not _SIDE_PENDING:
            torch.autograd.Variable._execution_engine.queue_callback(join_side_streams)
        _SIDE_PENDING.append(ev)
        return (dx.reshape(x3.shape), dctx.reshape(c3.shape), None, None, None, None, None, None, None, None,
                d_ln1_w, d_ln1_b, d_wq, d_wkv, d_wo, d_bo, d_ln2_w, d_ln2_b, d_w1, d_b1, d_w2, d_b2, d_lnf_w, d_lnf_b)


def ctypes_ptr_array(tensors):
    import ctypes as C
    return (C.c_void_p * len(tensors))(*[t.data_ptr() for t in tensors])


def encoder_supported(dim, inner, mlp):
    return os.environ.get("TMF_ENC_FUSED", "1") != "0" and bool(L.load().tmf_encoder_supported(int(dim), int(inner), int(mlp)))


def encoder(x, context, heads, scale, add_input, eps1, eps2, epsf, params, pack_cache=None, tap=None):
    """The fused encoder; with an ``AttnTap`` it returns (y, dots, attn) (DESIGN section 3.8)."""
    return EncoderFunction.apply(x, context, heads, scale, add_input, eps1, eps2, epsf, pack_cache, tap, *params)


class TokenPoolFunction(torch.autograd.Function):
    """x (B,N,C) -> mean over N (B,C) and/or max over N (B,C) (first-maximum gradient routing)."""

    @staticmethod
    def forward(ctx, x, want_mean, want_max):
        x = _f32c(x)
        B, N, C = x.shape
        mean = torch.empty((B, C), dtype=torch.float32, device=x.device) if want_mean else None
        mx = torch.empty((B, C), dtype=torch.float32, device=x.device) if want_max else None
        amax = torch.empty((B, C), dtype=torch.int32, device=x.device) if want_max else None
        L.call("tmf_token_pool_fwd", L.ptr(x), L.ptr(mean), L.ptr(mx), L.ptr(amax), B, N, C)
        ctx.shape, ctx.amax = (B, N, C), amax
        ctx.want = (want_mean, want_max)
        if want_mean and want_max:
            return mean, mx
        return mean if want_mean else mx

    @staticmethod
    def backward(ctx, *g):
        B, N, C = ctx.shape
        want_mean, want_max = ctx.want
        if want_mean and want_max:
            dmean, dmax = g
        elif want_mean:
            dmean, dmax = g[0], None
        else:
            dmean, dmax = None, g[0]
        dmean = _f32c(dmean) if dmean is not None else None
        dmax = _f32c(dmax) if dmax is not None else None
        dx = torch.empty((B, N, C), dtype=torch.float32, device=(dmean if dmean is not None else dmax).device)
        L.call("tmf_token_pool_bwd", L.ptr(dmean), L.ptr(dmax), L.ptr(ctx.amax), L.ptr(dx), B, N, C, 0)
        return dx, None, None


def token_pool(x, want_mean=True, want_max=True):
    return TokenPoolFunction.apply(x, want_mean, want_max)


class GradientReversalFunction(torch.autograd.Function):
    """reference models/gradient_reversal/functional.py:4-19: identity forward, -alpha * grad backward."""

    @staticmethod
    def forward(ctx, x, alpha):
        if torch.is_tensor(alpha):
            if alpha.is_cuda:
                ctx.alpha_dev, ctx.alpha = alpha.detach().reshape(-1).float(), 1.0
            else:
                ctx.alpha_dev, ctx.alpha = None, float(alpha.reshape(-1)[0])
        else:
            ctx.alpha_dev, ctx.alpha = None, float(alpha)
        return x.view_as(x)

    @staticmethod
    def backward(ctx, g):
        if not ctx.needs_input_grad[0]:
            return None, None
        g = _f32c(g)
        out = torch.empty_like(g)
        L.call("tmf_scale", L.ptr(g), L.ptr(out), -ctx.alpha, L.ptr(ctx.alpha_dev), g.numel())
        return out, None


def revgrad(x, alpha):
    return GradientReversalFunction.apply(x, alpha)


# ==============================================================================================================
# Grad-CAM   (csrc/gradcam.cu)
# ==============================================================================================================
def gradcam(acts, grads, size=None, normalize=True):
    """Grad-CAM maps of one or more towers' block activations ``acts`` and their gradients ``grads`` (fp32, logical
    (B,C,d,h,w)): ReLU(sum_c mean_p(G)[c] * A[c]), trilinearly upsampled to ``size`` = (D,H,W) when given
    (``F.interpolate(mode="trilinear", align_corners=False)``), normalised per sample to [0,1] when ``normalize``.
    Returns one fp32 (B,1,D,H,W) (or (B,1,d,h,w)) map per tower; both towers of a pair run in one launch sequence."""
    A = [_f32c(a.detach().permute(0, 2, 3, 4, 1)) for a in acts]
    G = [_f32c(g.detach().permute(0, 2, 3, 4, 1)) for g in grads]
    B, d, h, w, C = A[0].shape
    if any(t.shape != A[0].shape for t in A + G):
        raise ValueError("gradcam: every activation and gradient must have the same shape")
    D, H, W = tuple(size) if size is not None else (d, h, w)
    ups = int(size is not None)
    dev = A[0].device
    cams = [torch.empty((B, 1, D, H, W), dtype=torch.float32, device=dev) for _ in A]
    for i in range(0, len(A), 2):
        ng = min(2, len(A) - i)
        nws = int(L.load().tmf_gradcam_workspace_bytes(ng, B, d, h, w, C, D, H, W, ups, int(normalize)))
        if nws < 0:
            raise ValueError(f"gradcam: unsupported problem B={B} {d}x{h}x{w} C={C} -> {D}x{H}x{W}")
        ws = torch.empty(nws, dtype=torch.uint8, device=dev)
        L.call("tmf_gradcam", ng, L.ptrs(A[i:i + ng]), L.ptrs(G[i:i + ng]), L.ptrs(cams[i:i + ng]), B, d, h, w, C, D, H, W,
               ups, int(normalize), L.ptr(ws), nws)
    return cams


# ==============================================================================================================
# Layer-wise relevance propagation   (csrc/lrp.cu, csrc/conv1_dgrad.cu; DESIGN section 3.9)
# ==============================================================================================================
LRP_RULES = {"epsilon": L.LRP_EPSILON, "zplus": L.LRP_ZPLUS}


class LrpFold:
    """One conv layer's eval-mode BatchNorm fold for an LRP rule (``tmf_lrp_fold_pack``): the bf16 forward pack ``wf`` (the
    z+ convolution; rule zplus only), the bf16 dgrad pack ``wd`` (layers 1-6), the fp32 weight ``w32`` (layer 0) and the folded
    bias.  Rebuilt on the signature ``EvalFold`` uses: parameter / running-statistics addresses and versions and the epoch."""

    def __init__(self):
        self.sig = None
        self.wf = self.wd = self.w32 = self.bias = None

    def refresh(self, l, rule, tensors, bn_eps):
        w = tensors[0]
        sig = (_PARAM_EPOCH[0],) + tuple((t.data_ptr(), t._version) for t in tensors)
        if self.bias is None or self.bias.device != w.device:
            cout, cin, k = w.shape[0], w.shape[1], w.shape[2]
            self.bias = torch.empty(cout, dtype=torch.float32, device=w.device)
            if l == 0:
                self.w32 = torch.empty_like(w)
            else:
                self.wd = torch.empty((k ** 3, cin, cout), dtype=torch.bfloat16, device=w.device)
                if rule == L.LRP_ZPLUS:
                    self.wf = torch.empty((k ** 3, cout, cin), dtype=torch.bfloat16, device=w.device)
            self.sig = None
        if sig == self.sig:
            return
        cout, cin, k = w.shape[0], w.shape[1], w.shape[2]
        L.call("tmf_lrp_fold_pack", 1, *[L.ptrs([t]) for t in tensors], L.ptrs([self.wf]), L.ptrs([self.wd]),
               L.ptrs([self.w32]), L.ptrs([self.bias]), cout, cin, k, float(bn_eps), rule)
        self.sig = sig


def lrp_conv1_impl(B, D, H, W, cout, ng=1):
    """The block-1 LRP implementation ``tmf_lrp_conv1`` takes for this problem: ``L.CONV_UMMA`` (tcgen05) or
    ``L.CONV_DIRECT`` (CUDA cores: ``TMF_CONV_IMPL=direct``, rows wider than 128 voxels, Cout != 32)."""
    return int(L.load().tmf_lrp_conv1_impl(ng, conv_impl(), B, D, H, W, cout))


def lrp_towers(spec, hyper, folds, layer_params, kept, seeds, rule="epsilon", eps=1e-6):
    """LRP sweep, layer 6 down to 0, through one or two towers of the same shape in one launch sequence.

    ``folds[t]``: 7 ``LrpFold`` of tower t (cached by the caller); ``layer_params[t][l]``: (conv.weight, conv.bias, bn.weight,
    bn.bias, running_mean, running_var); ``kept[t]``: the 7 (input activation, y) pairs the folded eval forward kept (layer 0:
    the fp32 (B,1,D,H,W) volume); ``seeds[t]``: (a_T, g_T), fp32 (B,d,h,w,C) contiguous, whose product is the relevance at the
    tower output.  Returns (maps, totals): per tower an fp32 (B,1,D,H,W) relevance map and an fp32 (B, 8) tensor of per-sample
    relevance sums (the tower output, then entering layers 6 .. 0)."""
    rc = LRP_RULES[rule]
    ng = len(kept)
    impl = conv_impl()
    x = [k[0][0] for k in kept]
    B, _, D, H, W = x[0].shape
    dev = x[0].device
    totals = list(torch.empty((ng, B, 8), dtype=torch.float32, device=dev).unbind(0))
    c = None
    for l in range(len(spec.layers) - 1, -1, -1):
        cin, cout, ks, pool = spec.layers[l]
        bn_eps, _, slope = hyper[l]
        for t in range(ng):
            folds[t][l].refresh(l, rc, layer_params[t][l], bn_eps)
        fl = [folds[t][l] for t in range(ng)]
        act = [k[l][0] for k in kept]
        y = [k[l][1] for k in kept]
        Dl, Hl, Wl = y[0].shape[1:4]
        zp = None
        if rc == L.LRP_ZPLUS:
            zp = [torch.empty_like(v) for v in y]
            zero = torch.zeros(cout, dtype=torch.float32, device=dev)
            if l == 0:
                L.call("tmf_conv1_fwd", ng, L.ptrs(act), L.ptrs([f.w32 for f in fl]), L.ptrs([zero] * ng), L.ptrs(zp),
                       L.ptrs(None), B, Dl, Hl, Wl, cout, impl)
            else:
                L.call("tmf_conv3d_fwd", ng, L.ptrs(act), L.ptrs([f.wf for f in fl]), L.ptrs([zero] * ng), L.ptrs(zp),
                       L.ptrs(None), B, Dl, Hl, Wl, cin, cout, ks, impl, tag=f"tmf_conv3d_fwd@L{l}")
        if l == 0:
            a1 = [k[1][0] for k in kept]
            rx = [torch.empty((B, 1, D, H, W), dtype=torch.float32, device=dev) for _ in range(ng)]
            nws = int(L.load().tmf_lrp_conv1_workspace_bytes(ng, impl, B, D, H, W, cout))
            ws = torch.empty(nws, dtype=torch.uint8, device=dev)
            L.call("tmf_lrp_conv1", ng, L.ptrs(a1), L.ptrs(c), L.ptrs(y), L.ptrs(zp), L.ptrs([f.w32 for f in fl]), L.ptrs(x),
                   L.ptrs(rx), L.ptrs(totals), B, D, H, W, cout, float(eps), impl, L.ptr(ws), nws)
            return rx, totals
        if l == len(spec.layers) - 1:
            up_a, up_c, up32, col = [s[0] for s in seeds], [s[1] for s in seeds], 1, 0
        else:
            up_a, up_c, up32, col = [k[l + 1][0] for k in kept], c, 0, len(spec.layers) - 1 - l
        s = [torch.empty_like(v) for v in y]
        nws = int(L.load().tmf_lrp_ratio_workspace_bytes(ng, B, Dl, Hl, Wl, cout, pool))
        ws = torch.empty(nws, dtype=torch.uint8, device=dev)
        L.call("tmf_lrp_ratio", ng, L.ptrs(up_a), L.ptrs(up_c), up32, L.ptrs(y), L.ptrs(zp), L.ptrs(s), L.ptrs(totals), col,
               B, Dl, Hl, Wl, cout, pool, float(slope), float(eps), L.ptr(ws), nws, tag=f"tmf_lrp_ratio@L{l}")
        c = [torch.empty((B, Dl, Hl, Wl, cin), dtype=torch.bfloat16, device=dev) for _ in range(ng)]
        L.call("tmf_conv3d_fwd", ng, L.ptrs(s), L.ptrs([f.wd for f in fl]), L.ptrs(None), L.ptrs(c), L.ptrs(None),
               B, Dl, Hl, Wl, cout, cin, ks, impl, tag=f"tmf_conv3d_dgrad@L{l}")


def lrp_normalize(maps):
    """Divide each sample of each fp32 (B,1,D,H,W) map by its max |R|, in place (a map that is zero stays zero)."""
    for i in range(0, len(maps), 2):
        grp = maps[i:i + 2]
        B = grp[0].shape[0]
        L.call("tmf_lrp_normalize", len(grp), L.ptrs(grp), B, grp[0].numel() // B)
    return maps


# ==============================================================================================================
# Integrated gradients   (csrc/ig.cu; DESIGN section 3.10)
# ==============================================================================================================
def ig_block1(xs, folds, tensors, bn_eps):
    """Block 1 of one or two towers, once for a whole integrated-gradients path: the layer-0 ``EvalFold`` brought up to date
    (``tensors`` as for ``refresh_eval_folds``), u' = W' * x without bias (bf16 [B,D,H,W,C]) and umax = u' at the first
    maximum of each 2x2x2 window (bf16 [B,D/2,H/2,W/2,C]).  xs: fp32 contiguous (B,1,D,H,W) volumes."""
    refresh_eval_folds(folds, 0, tensors, bn_eps)
    ng = len(xs)
    B, _, D, H, W = xs[0].shape
    C = folds[0].bias.shape[0]
    dev = xs[0].device
    u = [torch.empty((B, D, H, W, C), dtype=torch.bfloat16, device=dev) for _ in range(ng)]
    zero = torch.zeros(C, dtype=torch.float32, device=dev)
    L.call("tmf_conv1_fwd", ng, L.ptrs(xs), L.ptrs([f.w32 for f in folds]), L.ptrs([zero] * ng), L.ptrs(u), L.ptrs(None),
           B, D, H, W, C, conv_impl())
    umax = [torch.empty((B, D // 2, H // 2, W // 2, C), dtype=torch.bfloat16, device=dev) for _ in range(ng)]
    pooled = [torch.empty_like(m) for m in umax]
    # identity coefficients and slope 1: the pass pools u' itself, and ymax is u' at the first maximum
    L.call("tmf_bn_act_pool_fwd_keepmax", ng, L.ptrs(u), L.ptrs([f.ident for f in folds]), L.ptrs(pooled), L.ptrs(umax), 0,
           B, D, H, W, C, 1.0)
    return u, umax


def ig_expand(umax, bias, alpha, slope):
    """The block-1 outputs at the path points ``alpha`` (fp32 device table of n): per tower (bf16 twin, fp32 value), both
    [n*B, D/2, H/2, W/2, C] step-major."""
    ng, n = len(umax), alpha.numel()
    B, C = umax[0].shape[0], umax[0].shape[-1]
    shape = (n * B,) + tuple(umax[0].shape[1:])
    a16 = [torch.empty(shape, dtype=torch.bfloat16, device=umax[0].device) for _ in range(ng)]
    a32 = [torch.empty(shape, dtype=torch.float32, device=umax[0].device) for _ in range(ng)]
    L.call("tmf_ig_expand", ng, L.ptrs(umax), L.ptrs(bias), L.ptr(alpha), n, L.ptrs(a16), L.ptrs(a32), B,
           umax[0].numel() // B, C, float(slope))
    return a16, a32


def ig_combine(grads, umax, bias, alpha, w, G, slope):
    """G[t] += sum_k w_k * grads[t][k*B + b] * LeakyReLU'(alpha_k * umax + b'), k in order (``tmf_ig_combine``); grads: fp32
    [n*B, D/2, H/2, W/2, C] contiguous, step-major."""
    ng, n = len(umax), alpha.numel()
    B, C = umax[0].shape[0], umax[0].shape[-1]
    L.call("tmf_ig_combine", ng, L.ptrs(grads), L.ptrs(umax), L.ptrs(bias), L.ptr(alpha), L.ptr(w), n, L.ptrs(G), B,
           umax[0].numel() // B, C, float(slope))


def ig_input_grad(G, u, folds, impl=None):
    """W'^T route(G): the block-1 input-gradient kernel with identity coefficients, zero bcoef and slope 1, fed bf16(G) and
    u' -- its dz is then G at the first maximum of u' in every window.  Returns fp32 (B,1,D,H,W) per tower."""
    ng = len(G)
    B, D, H, W, C = u[0].shape
    dev = G[0].device
    g16 = [torch.empty(g.shape, dtype=torch.bfloat16, device=dev) for g in G]
    L.call("tmf_narrow_f32", ng, L.ptrs(G), L.ptrs(g16), G[0].numel())
    bcoef = [torch.zeros(2 * C, dtype=torch.float32, device=dev)] * ng
    dx = [torch.empty((B, 1, D, H, W), dtype=torch.float32, device=dev) for _ in range(ng)]
    impl = conv_impl() if impl is None else impl
    nws = int(L.load().tmf_conv1_dgrad_fused_workspace_bytes(ng, impl, B, D, H, W, C))
    ws = torch.empty(nws, dtype=torch.uint8, device=dev) if nws > 0 else None
    L.call("tmf_conv1_dgrad_fused", ng, L.ptrs(g16), L.ptrs(u), L.ptrs([f.ident for f in folds]), L.ptrs(bcoef),
           L.ptrs([f.w32 for f in folds]), L.ptrs(dx), B, D, H, W, C, 1.0, impl, L.ptr(ws), nws)
    return dx


def ig_attribute(xs, dx):
    """dx[t] *= xs[t] in place (fp32 (B,1,D,H,W)); returns per tower the (B,) per-sample sums of the products."""
    ng = len(xs)
    B = xs[0].shape[0]
    per = xs[0].numel() // B
    sums = torch.empty((ng, B, 8), dtype=torch.float32, device=xs[0].device)
    nws = int(L.load().tmf_ig_attribute_workspace_bytes(ng, B, per))
    ws = torch.empty(nws, dtype=torch.uint8, device=xs[0].device)
    L.call("tmf_ig_attribute", ng, L.ptrs(xs), L.ptrs(dx), L.ptrs(list(sums.unbind(0))), B, per, L.ptr(ws), nws)
    return list(sums[:, :, 0].unbind(0))


# ==============================================================================================================
# Occlusion sensitivity with incremental recomputation   (csrc/occlusion.cu; DESIGN section 3.11)
# ==============================================================================================================
def occ_positions(E, w, s):
    """Window starts along an axis of extent E: i*s for i = 0 .. (E - w) // s (captum's ``Occlusion``)."""
    return list(range(0, E - w + 1, s))


class OccPlan:
    """Crop geometry of incremental occlusion through one sNet (host only, per axis; a window's geometry is the product of its
    three axes' entries).

    For layer l (0 .. 6) and every window: the changed region of the layer's input (layer 0: the window itself, then the
    recomputed output of layer l-1), the recompute region R of the layer's conv output (the changed outputs -- the changed input
    grown by the conv halo -- widened to whole 2x2x2 pooling windows at pooled layers) and the input crop, of one extent per layer
    for all windows: it covers R plus the halo, is shifted inward at the volume faces and starts on an even index at pooled
    layers, so that the crop's pooling grid is the global one.  Entry 7 is the tower output (the whole extent).

    ``crop[l]``: (Dc, Hc, Wc) of layer l's input crop (7: the output extent); ``full[l]``: the layer's full input extent;
    ``tab[l]``: int32 numpy [nwin, 3, 4], per window and axis (origin of the crop, lo, hi of the changed input region -- global
    coordinates of layer l's input --, origin of layer l-1's recomputed output in those coordinates); window n = (i*nH + j)*nW + k.
    """

    def __init__(self, dims, window, stride, layers):
        import numpy as np
        self.dims, self.window, self.stride = tuple(dims), tuple(window), tuple(stride)
        self.grid = tuple(len(occ_positions(E, w, s)) for E, w, s in zip(dims, window, stride))
        axes = [self._axis(E, [(a, a + w) for a in occ_positions(E, w, s)], layers) for E, w, s in zip(dims, window, stride)]
        self.crop = [tuple(ax[0][l] for ax in axes) for l in range(len(layers) + 1)]
        self.full = [tuple(ax[1][l] for ax in axes) for l in range(len(layers) + 1)]
        nD, nH, nW = self.grid
        self.tab = []
        for l in range(len(layers) + 1):
            t = np.empty((nD, nH, nW, 3, 4), dtype=np.int32)
            t[:, :, :, 0] = axes[0][2][:, l].reshape(nD, 1, 1, 4)
            t[:, :, :, 1] = axes[1][2][:, l].reshape(1, nH, 1, 4)
            t[:, :, :, 2] = axes[2][2][:, l].reshape(1, 1, nW, 4)
            self.tab.append(t.reshape(nD * nH * nW, 3, 4))

    @property
    def nwin(self):
        return self.grid[0] * self.grid[1] * self.grid[2]

    @staticmethod
    def _axis(E, spans, layers):
        """One axis for the intervals ``spans`` [(a, b)] of the input changed, one per window or box: crop extents (one per
        layer for all of them), full extents and the [n, 8, 4] table (crop origin, lo, hi, previous output origin)."""
        import numpy as np
        nl = len(layers)
        ext = [E]
        for ks, pool in layers:
            ext.append(ext[-1] // 2 if pool != L.POOL_NONE else ext[-1])
        # pass 1: per window and layer the changed input [a, b), the recompute region [ra, rb) and the needed input [na, nb)
        geo = []
        for a, b in spans:
            rows = []
            for l, (ks, pool) in enumerate(layers):
                e, h = ext[l], ks // 2
                oa, ob = max(a - h, 0), min(b + h, e)                     # conv outputs that change
                if pool != L.POOL_NONE:
                    ra, rb = oa - oa % 2, min(ob + ob % 2, e - e % 2)     # whole pooling windows (floor mode drops e-1)
                else:
                    ra, rb = oa, ob
                rows.append((a, b, ra, rb, max(ra - h, 0), min(rb + h, e)))
                a, b = (ra // 2, rb // 2) if pool != L.POOL_NONE else (ra, rb)
            rows.append((a, b))
            geo.append(rows)
        crop = []
        for l, (ks, pool) in enumerate(layers):
            e, even = ext[l], pool != L.POOL_NONE
            c = max(r[l][5] - (r[l][4] - r[l][4] % 2 if even else r[l][4]) for r in geo)
            if even and c < e and (e - c) % 2:
                c += 1                           # the inward shift at the far face must keep an even origin
            crop.append(min(c, e))
        crop.append(ext[nl])
        tab = np.zeros((len(spans), nl + 1, 4), dtype=np.int32)
        for n, rows in enumerate(geo):
            prev = 0
            for l, (ks, pool) in enumerate(layers):
                e, h, c = ext[l], ks // 2, crop[l]
                a, b, ra, rb, na, nb = rows[l]
                c0 = min(na - na % 2 if pool != L.POOL_NONE else na, e - c)
                assert c0 >= 0 and (pool == L.POOL_NONE or c0 % 2 == 0), (l, c0)
                assert c0 <= na and nb <= c0 + c and c0 <= a and b <= c0 + c, (l, c0, c, rows[l])
                # a crop output within h of a crop face that is not a volume face saw zero padding instead of data
                lo_ok, hi_ok = c0 + (h if c0 > 0 else 0), c0 + c - (h if c0 + c < e else 0)
                assert lo_ok <= ra and rb <= hi_ok, (l, c0, c, ra, rb)
                tab[n, l] = (c0, a, b, prev)
                prev = c0 // 2 if pool != L.POOL_NONE else c0
            a, b = rows[nl]
            tab[n, nl] = (0, a, b, prev)
            # the changed input of every layer lies inside the previous layer's recomputed output
            for l in range(1, nl + 1):
                ks, pool = layers[l - 1]
                pc = crop[l - 1] // 2 if pool != L.POOL_NONE else crop[l - 1]
                assert tab[n, l, 3] <= tab[n, l, 1] and tab[n, l, 2] <= tab[n, l, 3] + pc, (l, tab[n, l])
        return crop, ext, tab

    def out_extent(self, l, pool):
        """Extent of layer l's recomputed (pooled) crop output."""
        return tuple(c // 2 for c in self.crop[l]) if pool != L.POOL_NONE else self.crop[l]


def occ_pass_limit(plan, spec, B, ng):
    """Most windows one pass may take (rows m*B) while every crop launch stays inside its kernel's 32-bit index limits:
    tmf_conv1_fwd rows*D*H*W < 2^31, tmf_bn_act_pool_fwd rows*D*H*W*C/8 < 2^31 and the column conv rows*NC*D < 2^30 (NC from
    its launch plan, counted wherever the plan exists)."""
    import ctypes
    per = []
    for l, (cin, cout, ks, pool) in enumerate(spec.layers):
        Dc, Hc, Wc = plan.crop[l]
        vox = B * Dc * Hc * Wc
        per.append((vox * (cout // 8), 1 << 31))
        if l == 0:
            per.append((vox, 1 << 31))
        else:
            info = (ctypes.c_int * 6)()
            if L.load().tmf_conv3d_col_plan_info(ng, Dc, Hc, Wc, cin, cout, ks, info) == 0:
                per.append((B * info[3] * Dc, 1 << 30))
    return max(1, min((lim - 1) // c for c, lim in per))


def occ_input(xs, tab, m, baseline, extent):
    """fp32 (m*B, 1, Dc, Hc, Wc) layer-0 crops per tower (``tmf_occ_input``); xs: fp32 contiguous (B,1,D,H,W)."""
    B, _, D, H, W = xs[0].shape
    out = [torch.empty((m * B, 1) + tuple(extent), dtype=torch.float32, device=xs[0].device) for _ in xs]
    L.call("tmf_occ_input", len(xs), L.ptrs(xs), L.ptr(tab), m, float(baseline), L.ptrs(out), B, D, H, W, *extent)
    return out


def occ_compose(base, crops, tab, m, extent, out=None, tag=None):
    """Input crops (m*B, Dc, Hc, Wc, C) per tower (``tmf_occ_compose``): base (B, D, H, W, C) contiguous, bf16 or fp32; crops:
    the previous layer's recomputed outputs (m*B, Dp, Hp, Wp, C), or None to replicate the base; ``out``: optional contiguous
    destinations."""
    B, D, H, W, C = base[0].shape
    if out is None:
        out = [torch.empty((m * B,) + tuple(extent) + (C,), dtype=base[0].dtype, device=base[0].device) for _ in base]
    Dp, Hp, Wp = crops[0].shape[1:4] if crops is not None else (0, 0, 0)
    L.call("tmf_occ_compose", len(base), L.ptrs(base), L.ptrs(crops), L.ptr(tab), m, L.ptrs(out), B, D, H, W, *extent,
           Dp, Hp, Wp, C, int(base[0].dtype == torch.float32), tag=tag)
    return out


def occ_layer(l, spec, hyper, folds, act, extent, impl):
    """Layer l of the folded eval sNet on a batch of crops, as ``SNetFunction._eval_forward`` runs it: the conv on the folded
    operands, then LeakyReLU and the pool with the identity coefficients.  act: fp32 (R,1,D,H,W) crops at layer 0, else bf16
    (R,D,H,W,Cin); returns (R, pooled extent, Cout), fp32 at the last layer."""
    cin, cout, ks, pool = spec.layers[l]
    slope = hyper[l][2]
    R = act[0].shape[0]
    dev = act[0].device
    y = [torch.empty((R,) + tuple(extent) + (cout,), dtype=torch.bfloat16, device=dev) for _ in act]
    bias = [fo.bias for fo in folds]
    if l == 0:
        L.call("tmf_conv1_fwd", len(act), L.ptrs(act), L.ptrs([fo.w32 for fo in folds]), L.ptrs(bias), L.ptrs(y), L.ptrs(None),
               R, *extent, cout, impl, tag="tmf_conv1_fwd@occ")
    else:
        L.call("tmf_conv3d_fwd", len(act), L.ptrs(act), L.ptrs([fo.wf for fo in folds]), L.ptrs(bias), L.ptrs(y), L.ptrs(None),
               R, *extent, cin, cout, ks, impl, tag=f"tmf_conv3d_fwd@occL{l}")
    last = l == len(spec.layers) - 1
    Do, Ho, Wo = _pooled(*extent, pool)
    out = [torch.empty((R, Do, Ho, Wo, cout), dtype=torch.float32 if last else torch.bfloat16, device=dev) for _ in act]
    L.call("tmf_bn_act_pool_fwd", len(act), L.ptrs(y), L.ptrs([fo.ident for fo in folds]), L.ptrs(out), int(last), R, *extent,
           cout, pool, slope, tag=f"tmf_bn_act_pool_fwd@occL{l}")
    return out


def occ_towers(spec, hyper, folds, xs, kept, base_out, plan, tabs, m, baseline, out):
    """One pass of m windows through one or two towers of the same shape: the layer-0 crops, then per layer the conv on the
    crops and the composition of the next layer's input crops from the recomputed region and the kept base activations;
    the final composition writes the (m*B, d, h, w, C) fp32 tower outputs into ``out``.  folds[t]: the tower's 7 ``EvalFold``
    (current: the base forward refreshed them); kept[t]: its 7 (input activation, y) pairs; base_out[t]: its fp32 (B,d,h,w,C)
    output; tabs: the pass's device tables (``OccPlan.tab`` rows), one per layer and the output."""
    return occ_crops(spec, hyper, folds, occ_input(xs, tabs[0], m, baseline, plan.crop[0]), kept, base_out, plan, tabs, m, out)


def occ_crops(spec, hyper, folds, act, kept, base_out, plan, tabs, m, out):
    """``occ_towers`` from given fp32 (m*B, 1, Dc, Hc, Wc) layer-0 crops ``act`` (one per tower): layers 0 .. 6 and the
    composition of the tower outputs into ``out``.  ``plan``: an ``OccPlan`` or a ``BoxPlan``."""
    impl = conv_impl()
    for l in range(len(spec.layers)):
        if l > 0:
            act = occ_compose([k[l][0] for k in kept], act, tabs[l], m, plan.crop[l], tag=f"tmf_occ_compose@L{l}")
        act = occ_layer(l, spec, hyper, [f[l] for f in folds], act, plan.crop[l], impl)
    return occ_compose(base_out, act, tabs[-1], m, plan.crop[-1], out=out, tag="tmf_occ_compose@out")


def occ_map(scores, plan):
    """Per tower, the fp32 (B,1,D,H,W) map: each voxel's mean score over the windows containing it (``tmf_occ_map``).
    scores: fp32 contiguous (B, nD, nH, nW) per tower."""
    B = scores[0].shape[0]
    maps = [torch.empty((B, 1) + plan.dims, dtype=torch.float32, device=scores[0].device) for _ in scores]
    for i in range(0, len(scores), 2):
        L.call("tmf_occ_map", len(scores[i:i + 2]), L.ptrs(scores[i:i + 2]), L.ptrs(maps[i:i + 2]), B, *plan.dims, *plan.grid,
               *plan.window, *plan.stride)
    return maps


# ==============================================================================================================
# Feature ablation over regions of a mask, with incremental recomputation   (csrc/ablation.cu; DESIGN section 3.12)
# ==============================================================================================================
# Extent classes: per axis, a feature's box extent rounds up to the first rung that is at least as large (the full extent past
# the last rung).  The features of one class share crop extents, the largest over the class.  Coarse rungs: fewer, fuller
# passes through the fusion stack outweigh the padding (finer ladders measured slower, DESIGN section 3.12).
ABL_LADDER = (24, 48, 96)


class BoxPlan:
    """Crop geometry of incremental recomputation for a list of boxes ``[((a0, b0), (a1, b1), (a2, b2))]`` of the input, one
    per feature of an extent class (host only).  Each axis goes through ``OccPlan._axis`` with the boxes' intervals, so the
    crop extents are one per layer for all the boxes; ``crop`` and ``full`` as for ``OccPlan``; ``tab[l]``: int32 numpy
    [n, 3, 4], per box and axis, the same layout; ``ids``: int32 numpy [n], the boxes' feature ids."""

    def __init__(self, dims, boxes, layers, ids):
        import numpy as np
        self.dims = tuple(dims)
        axes = [OccPlan._axis(E, [bx[a] for bx in boxes], layers) for a, E in enumerate(self.dims)]
        self.crop = [tuple(ax[0][l] for ax in axes) for l in range(len(layers) + 1)]
        self.full = [tuple(ax[1][l] for ax in axes) for l in range(len(layers) + 1)]
        self.tab = [np.ascontiguousarray(np.stack([ax[2][:, l] for ax in axes], axis=1)) for l in range(len(layers) + 1)]
        self.ids = np.asarray(ids, dtype=np.int32)

    @property
    def n(self):
        return len(self.ids)


def abl_boxes(mask, F):
    """Bounding box of every id 0 .. F-1 of an integer mask (1|B, 1, D, H, W), over all its samples (torch ops on the mask's
    device, then one device-to-host copy): int64 numpy [F, 6] (lo_D, lo_H, lo_W, hi_D, hi_H, hi_W), hi exclusive; an absent
    id has lo = extent and hi = 0."""
    dims = mask.shape[2:]
    ids = mask.reshape(-1).long()
    cols = []
    for a, E in enumerate(dims):
        shape = [1] * 5
        shape[2 + a] = E
        c = torch.arange(E, device=mask.device).view(shape).expand(mask.shape).reshape(-1)
        cols.append((torch.full((F,), E, dtype=torch.long, device=mask.device).scatter_reduce_(0, ids, c, "amin"),
                     torch.full((F,), -1, dtype=torch.long, device=mask.device).scatter_reduce_(0, ids, c, "amax") + 1))
    return torch.stack([lo for lo, _ in cols] + [hi for _, hi in cols], 1).cpu().numpy()


def abl_classes(boxes, dims):
    """The present features of ``abl_boxes`` grouped by extent class (``ABL_LADDER``): [(class key, [ids ascending])] in key
    order.  The grouping depends on the mask alone, so a feature's crop extents do not depend on how the passes are cut."""
    classes = {}
    for f in range(len(boxes)):
        ext = [int(boxes[f, 3 + a] - boxes[f, a]) for a in range(3)]
        if ext[0] <= 0:
            continue
        key = tuple(next((r for r in ABL_LADDER if e <= r < E), E) for e, E in zip(ext, dims))
        classes.setdefault(key, []).append(f)
    return sorted(classes.items())


def abl_plan(boxes, ids, dims, layers):
    """The ``BoxPlan`` of one extent class: the features ``ids`` with their boxes from ``abl_boxes``."""
    return BoxPlan(dims, [tuple((int(boxes[f, a]), int(boxes[f, 3 + a])) for a in range(3)) for f in ids], layers, ids)


def abl_input(xs, mask, baselines, tab, ids, m, extent):
    """fp32 (m*B, 1, Dc, Hc, Wc) layer-0 crops per tower (``tmf_abl_input``): x, with the baseline where the mask holds the
    row's feature id.  xs: fp32 contiguous (B,1,D,H,W); mask: int32 contiguous (1|B,1,D,H,W); baselines: per tower a float or
    an fp32 contiguous (1|B,1,D,H,W) tensor; tab: a pass's layer-0 rows of ``BoxPlan.tab``; ids: int32 [m], their features."""
    import ctypes
    B, _, D, H, W = xs[0].shape
    out = [torch.empty((m * B, 1) + tuple(extent), dtype=torch.float32, device=xs[0].device) for _ in xs]
    vols = [b if torch.is_tensor(b) else None for b in baselines]
    vals = (ctypes.c_float * len(xs))(*[0.0 if torch.is_tensor(b) else float(b) for b in baselines])
    per = sum(1 << g for g, v in enumerate(vols) if v is not None and v.shape[0] > 1)
    L.call("tmf_abl_input", len(xs), L.ptrs(xs), L.ptr(mask), int(mask.shape[0] > 1), L.ptrs(vols), vals, per, L.ptr(tab),
           L.ptr(ids), m, L.ptrs(out), B, D, H, W, *extent)
    return out


def abl_map(scores, mask):
    """Per tower, the fp32 (B,1,D,H,W) map with each voxel holding its feature's score, map[b, v] = scores[b, mask[b|0, v]]
    (``tmf_abl_map``).  scores: fp32 contiguous (B, F) per tower; mask: int32 contiguous (1|B,1,D,H,W), ids < F."""
    B, F = scores[0].shape
    dims = tuple(mask.shape[2:])
    maps = [torch.empty((B, 1) + dims, dtype=torch.float32, device=scores[0].device) for _ in scores]
    for i in range(0, len(scores), 2):
        L.call("tmf_abl_map", len(scores[i:i + 2]), L.ptrs(scores[i:i + 2]), L.ptr(mask), int(mask.shape[0] > 1), F,
               L.ptrs(maps[i:i + 2]), B, *dims)
    return maps


# ==============================================================================================================
# Shapley value sampling over regions of a mask, with per-chain state   (csrc/shapley.cu; DESIGN section 3.13)
# ==============================================================================================================
# Bytes of chain state (per chain: every tower's kept layer 1-6 inputs and its tower output, for all B samples) one group of
# permutations may hold; a call runs its permutations in groups that fit.  The chains are independent, so the grouping
# changes the memory and never a bit of the result.
SHAP_STATE_BYTES = 8 << 30


def shap_permutations(ids, n_samples):
    """``n_samples`` orders of the players ``ids`` (int64 numpy [F']): int64 (n_samples, F'), one ``torch.randperm(F')`` per
    row from torch's global CPU generator, as captum's ``ShapleyValueSampling`` draws them."""
    ids = torch.as_tensor(ids, dtype=torch.int64)
    return torch.stack([ids[torch.randperm(len(ids))] for _ in range(n_samples)])


def shap_schedule(perms, cls_of, caps):
    """Passes of the chains of ``perms`` (int numpy [P, F'], region ids): a pass takes chains whose next region is in one extent
    class -- the class with the most waiting chains, the smaller class index (``abl_classes`` order) on a tie -- in ascending
    chain order, at most ``caps[class]`` of them.  cls_of: {id: class index}.  Returns [(class, [(p, k)])]: every (p, k) once,
    each chain's steps in order, a chain at most once per pass.  Host only; depends on the permutations alone."""
    P, Fp = perms.shape
    nxt = [0] * P
    left = P * Fp
    passes = []
    while left:
        waiting = {}
        for p in range(P):
            if nxt[p] < Fp:
                waiting.setdefault(cls_of[int(perms[p, nxt[p]])], []).append(p)
        c = min(waiting, key=lambda c: (-len(waiting[c]), c))
        chains = waiting[c][:caps[c]]
        passes.append((c, [(p, nxt[p]) for p in chains]))
        for p in chains:
            nxt[p] += 1
        left -= len(chains)
    return passes


def shap_input(xs, mask, baselines, tab, rank, perm, step, m, extent):
    """fp32 (m*B, 1, Dc, Hc, Wc) layer-0 crops per tower (``tmf_shap_input``): x where the voxel's region comes at or before
    the row's step in the row's permutation, else the baseline.  xs, mask and baselines as for ``abl_input``; rank: int32
    contiguous (P, F); perm, step: int32 [m]."""
    import ctypes
    B, _, D, H, W = xs[0].shape
    out = [torch.empty((m * B, 1) + tuple(extent), dtype=torch.float32, device=xs[0].device) for _ in xs]
    vols = [b if torch.is_tensor(b) else None for b in baselines]
    vals = (ctypes.c_float * len(xs))(*[0.0 if torch.is_tensor(b) else float(b) for b in baselines])
    per = sum(1 << g for g, v in enumerate(vols) if v is not None and v.shape[0] > 1)
    L.call("tmf_shap_input", len(xs), L.ptrs(xs), L.ptr(mask), int(mask.shape[0] > 1), L.ptrs(vols), vals, per, L.ptr(tab),
           L.ptr(rank), rank.shape[1], L.ptr(perm), L.ptr(step), m, L.ptrs(out), B, D, H, W, *extent)
    return out


def shap_compose(state, sidx, crops, tab, m, extent, out=None, tag=None):
    """Input crops (m*B, Dc, Hc, Wc, C) per tower (``tmf_shap_compose``), composed as ``occ_compose`` composes them but from the
    rows' chain states, whose changed region is then overwritten with the crops'.  state: (S*B, D, H, W, C) contiguous, bf16 or
    fp32, per tower; sidx: int32 [m], distinct chain indices; crops: the previous layer's recomputed outputs."""
    C = state[0].shape[-1]
    D, H, W = state[0].shape[1:4]
    B = crops[0].shape[0] // m
    if out is None:
        out = [torch.empty((m * B,) + tuple(extent) + (C,), dtype=state[0].dtype, device=state[0].device) for _ in state]
    L.call("tmf_shap_compose", len(state), L.ptrs(state), L.ptr(sidx), L.ptrs(crops), L.ptr(tab), m, L.ptrs(out), B, D, H,
           W, *extent, *crops[0].shape[1:4], C, int(state[0].dtype == torch.float32), tag=tag)
    return out


def shap_crops(spec, hyper, folds, act, state, plan, tabs, sidx, m, out):
    """One step of m chains through one or two towers of the same shape, as ``occ_crops`` runs a pass, with the chain states in
    place of the base activations: state[t][l] (l = 1 .. 6: the kept layer input, 7: the fp32 tower output), (S*B, ...) per
    tower; the composed tower outputs go to ``out`` and every state holds the step's result afterwards."""
    impl = conv_impl()
    for l in range(len(spec.layers)):
        if l > 0:
            act = shap_compose([s[l] for s in state], sidx, act, tabs[l], m, plan.crop[l], tag=f"tmf_shap_compose@L{l}")
        act = occ_layer(l, spec, hyper, [f[l] for f in folds], act, plan.crop[l], impl)
    return shap_compose([s[-1] for s in state], sidx, act, tabs[-1], m, plan.crop[-1], out=out, tag="tmf_shap_compose@out")
