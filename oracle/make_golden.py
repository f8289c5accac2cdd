"""Pin the oracle against the real reference and write the golden fixtures  --  TEST INFRASTRUCTURE ONLY.

Run in the authoring container (needs the read-only reference checkout):

    PYTHONDONTWRITEBYTECODE=1 python oracle/make_golden.py [--reference /root/reference]

For every case it
  1. instantiates the UNMODIFIED reference ``nn.Module`` (reference models/mymodel.py), loads procedural
     weights (``transmf_ad_b200.synthetic.procedural_state``) and runs forward + the caller's losses
     (reference kfold_train_adversarial.py:119-131) + backward on synthetic volumes;
  2. runs ``oracle/restatement.py`` on the same state / inputs and asserts bit-equality of outputs, every
     gradient and every BatchNorm buffer (this is what pins the restatement);
  3. stores outputs, losses, per-tensor gradient norms and strided gradient samples, and updated BN buffers
     in ``tests/golden/<case>.pt`` (small), plus the state-dict key/shape manifest in ``tests/golden/keys.json``.

``/root/reference`` does not exist on the GPU box; the fixtures are what travels.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle import restatement as R                      # noqa: E402
from transmf_ad_b200.synthetic import make_labels, make_volumes, procedural_state   # noqa: E402

CASES = {
    # name: (model, ctor kwargs, batch, volume shape, weight seed).  Models with BatchNorm1d heads use B = 8: with two or
    # three samples BatchNorm1d maps every feature to +-1 and turns rounding noise into O(1) logit changes.
    "model_ad_h4": ("model_ad", dict(dim=128, depth=3, heads=4, dim_head=32, mlp_dim=512, dropout=0.), 8, (35, 38, 33), 0),
    "model_ad_h8": ("model_ad", dict(dim=128, depth=3, heads=8, dim_head=16, mlp_dim=512, dropout=0.), 8, (32, 33, 34), 1),
    "model_cnn_ad": ("model_CNN_ad", dict(dim=128), 8, (33, 35, 34), 2),
    "model_single": ("model_single", dict(dim=128), 2, (34, 33, 37), 3),
    "model_transformer": ("model_transformer", dict(dim=128, depth=2, heads=4, dim_head=32, mlp_dim=256, dropout=0.), 8, (32, 32, 32), 4),
    "model_transformer_res": ("model_transformer_res", dict(dim=128, depth=2, heads=4, dim_head=32, mlp_dim=256, dropout=0.), 3, (32, 32, 32), 5),
    "model_cnn": ("model_CNN", dict(dim=128), 2, (32, 32, 32), 6),
    "model_ad_dim64": ("model_ad", dict(dim=64, depth=1, heads=2, dim_head=16, mlp_dim=96, dropout=0.), 8, (32, 36, 32), 7),
    # BASELINE configurations at the full 91x109x91 volume (SURVEY.md section 8d): C3 / C2 at batch 8, C1 at batch 2
    "model_ad_full_b8": ("model_ad", dict(dim=128, depth=3, heads=4, dim_head=32, mlp_dim=512, dropout=0.), 8, (91, 109, 91), 14),   # seed scanned: every train-mode margin > 0.3
    "model_cnn_ad_full_b8": ("model_CNN_ad", dict(dim=128), 8, (91, 109, 91), 9),
    "model_ad_full_b2": ("model_ad", dict(dim=128, depth=3, heads=4, dim_head=32, mlp_dim=512, dropout=0.), 2, (91, 109, 91), 10),
    # BASELINE configs[4]: the MiSePyNet baseline (reference models/MiSePyNet.py; its slice convolutions hard-code 91x109x91)
    "mnet_b4": ("Mnet", dict(), 4, (91, 109, 91), 11),
}
GRAD_SAMPLE = 48
# CPU threads of the fixture run.  The number of threads sets how torch splits the fp32 sums of the backward pass, and
# the gradients of a conv bias in front of a train-mode BatchNorm (zero up to rounding) and of the batch-2 full-size case
# follow that split; tests/test_oracle_golden.py recomputes the fixtures with the same count.
GOLDEN_THREADS = 8


def sample(t):
    f = t.detach().flatten()
    stride = max(1, f.numel() // GRAD_SAMPLE)
    return f[::stride][:GRAD_SAMPLE].clone()


def oracle_forward(kind, sd, inputs, kwargs, training, p_drop):
    heads = kwargs.get("heads", 4)
    if kind == "model_ad":
        return R.model_ad_forward(sd, *inputs, heads=heads, training=training, p_drop=p_drop)
    if kind == "model_CNN_ad":
        return R.model_cnn_ad_forward(sd, *inputs, training=training)
    if kind == "model_single":
        return (R.model_single_forward(sd, inputs[0], training=training),)
    if kind == "model_CNN":
        return (R.model_cnn_forward(sd, *inputs, training=training),)
    if kind == "model_transformer":
        return (R.model_transformer_forward(sd, *inputs, heads=heads, training=training, p_drop=p_drop),)
    if kind == "model_transformer_res":
        return (R.model_transformer_res_forward(sd, *inputs, heads=heads, training=training, p_drop=p_drop),)
    if kind == "Mnet":
        return (R.mnet_forward(sd, *inputs, training=training, p_drop=p_drop),)
    raise KeyError(kind)


def losses(outs, label):
    if len(outs) == 3:
        return R.adversarial_losses(outs[0], outs[1], outs[2], label)
    ce = torch.nn.functional.cross_entropy(outs[0], label)        # kfold_train_single.py:105
    return ce, torch.zeros(()), ce


def set_dropout(module, p):
    """Only the classifier-head Dropout(0.5) layers (mymodel.py:190-191); the transformer's stay at opt.dropout = 0."""
    for m in module.modules():
        if isinstance(m, torch.nn.Dropout):
            if not hasattr(m, "_p0"):
                m._p0 = m.p
            if m._p0 == 0.5:
                m.p = p


def run_case(name, refmods, outdir):
    kind, kwargs, B, shape, wseed = CASES[name]
    if kind == "Mnet":
        import models.MiSePyNet as mise           # the real reference baseline
        ref = mise.Mnet()
    else:
        ref = getattr(refmods, kind)(**kwargs)
    state = procedural_state(ref.state_dict(), seed=wseed)
    ref.load_state_dict(state)
    label = make_labels(B)
    mri = make_volumes(B, shape, seed=11 + wseed, labels=label)
    pet = make_volumes(B, shape, seed=23 + wseed, labels=label)
    inputs = (mri,) if kind == "model_single" else (mri, pet)

    gold = {"case": name, "kind": kind, "kwargs": kwargs, "batch": B, "shape": shape, "weight_seed": wseed,
            "input_seeds": (11 + wseed, 23 + wseed)}
    # ---- (A) dropout-on CPU check of the restatement only (CUDA cannot reproduce the CPU RNG stream) ----
    for p_drop, tag in ((0.5, "drop"), (0.0, "train")):
        ref.load_state_dict(state)
        ref.train()
        set_dropout(ref, p_drop)
        ref.zero_grad()
        torch.manual_seed(5)
        outs = ref(*inputs)
        outs = outs if isinstance(outs, tuple) else (outs,)
        ce, ad, total = losses(outs, label)
        total.backward()

        sd = R.clone_state(state)
        torch.manual_seed(5)
        o_outs = oracle_forward(kind, sd, inputs, kwargs, True, p_drop)
        o_ce, o_ad, o_total = losses(o_outs, label)
        o_total.backward()
        for a, b in zip(outs, o_outs):
            assert torch.equal(a, b), f"{name}/{tag}: oracle forward differs from the reference"
        assert torch.equal(total, o_total)
        ref_sd = ref.state_dict()
        for k, p in ref.named_parameters():
            if p.grad is None:                # dead parameters (Mnet: spatial_cnn.conv2 / conv3 are never called, MiSePyNet.py:89-94)
                assert sd[k].grad is None, k
                continue
            assert sd[k].grad is not None, k
            assert torch.equal(p.grad, sd[k].grad), f"{name}/{tag}: grad {k} differs"
        for k, v in ref_sd.items():
            if "running" in k or "num_batches" in k:
                assert torch.equal(v, sd[k]), f"{name}/{tag}: buffer {k} differs"
    # (the p=0 results are what we store)
    gold["train_outs"] = [o.detach().clone() for o in outs]
    gold["train_losses"] = (float(ce), float(ad), float(total))
    gold["grad_norm"] = {k: float(p.grad.norm()) for k, p in ref.named_parameters() if p.grad is not None}
    gold["grad_sample"] = {k: sample(p.grad) for k, p in ref.named_parameters() if p.grad is not None}
    gold["buffers_after"] = {k: v.clone() for k, v in ref.state_dict().items()
                             if "running" in k or "num_batches" in k}
    # ---- (B) eval-mode forward with the post-step buffers (val_step, kfold_train_adversarial.py:144-161) ----
    ref.eval()
    with torch.no_grad():
        e_outs = ref(*inputs)
    e_outs = e_outs if isinstance(e_outs, tuple) else (e_outs,)
    sd_eval = R.clone_state(ref.state_dict(), requires_grad=False)
    with torch.no_grad():
        oe = oracle_forward(kind, sd_eval, inputs, kwargs, False, 0.5)
    for a, b in zip(e_outs, oe):
        assert torch.equal(a, b), f"{name}: eval oracle differs"
    gold["eval_outs"] = [o.clone() for o in e_outs]
    gold["eval_argmax"] = e_outs[0].argmax(1)
    torch.save(gold, os.path.join(outdir, name + ".pt"))
    manifest = [[k, list(v.shape), str(v.dtype)] for k, v in ref.state_dict().items()]   # ordered
    print(f"[golden] {name}: ok  logits={outs[0].detach().flatten().tolist()[:4]} loss={float(total):.6f}")
    return kind + json.dumps(kwargs, sort_keys=True), manifest


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference", default="/root/reference")
    ap.add_argument("--out", default=os.path.join(ROOT, "tests", "golden"))
    ap.add_argument("--cases", nargs="*", default=list(CASES))
    args = ap.parse_args()
    sys.dont_write_bytecode = True
    sys.path.insert(0, args.reference)
    import models.mymodel as refmods           # the real reference
    os.makedirs(args.out, exist_ok=True)
    torch.set_num_threads(GOLDEN_THREADS)
    keys = {}
    kpath = os.path.join(args.out, "keys.json")
    if os.path.exists(kpath):
        with open(kpath) as f:
            keys = json.load(f)
    for name in args.cases:
        k, manifest = run_case(name, refmods, args.out)
        keys[k] = manifest
    with open(os.path.join(args.out, "keys.json"), "w") as f:
        json.dump(keys, f, indent=0)
    print("[golden] wrote", args.out)


if __name__ == "__main__":
    main()
