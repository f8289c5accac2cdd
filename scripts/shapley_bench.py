"""Shapley-value-sampling measurements on one GPU, in one process:

  1. interpret.shapley_sampling(model_ad) over a seeded synthetic atlas (chains with per-chain state: each step recomputes
     only what the added region's bounding box changes) against the brute-force loop a user writes by hand (one model call
     per pass on materialised composite volumes of the same permutations, one modality at a time), with the same volumes
     per pass, alternated three times: ms per call and subjects/s;
  2. the pass schedule: passes, mean chains per pass, and the chain-state bytes, computed from the shapes;
  3. one call under per-launch CUDA events: the crop launches and the fusion stack plus heads per pass, against the host
     time to enqueue the call (is the call launch-bound?);
  4. the worst score difference against brute force over max |f(x)|;
  5. the GPU name and power limit, read in the same run (nvidia-smi query only).

Usage: python scripts/shapley_bench.py [--batch 8] [--cells 96] [--samples 25] [--internal-batch 256] [--out FILE]
Defaults: model_ad in eval mode, B = 8 subjects of 91 x 109 x 91, 96 Voronoi cells plus background, baseline 0, 25
permutations drawn after torch.manual_seed(0).  A brute-force pass moves gigabytes, far beyond the 126 MB L2.
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from saliency_bench import SHAPE, gpu_info, model_ad, timed   # noqa: E402
from transmf_ad_b200 import _lib as L                         # noqa: E402
from transmf_ad_b200 import functional as TF                  # noqa: E402
from transmf_ad_b200.interpret import shapley_sampling        # noqa: E402
from transmf_ad_b200.synthetic import make_atlas              # noqa: E402


def brute_force(model, xs, target, mask, perms, baseline, chunk):
    """Scores (per tower, (B, F)) from the model's own forward on the materialised composite volumes of every chain of
    ``perms``, ``chunk`` chain steps of one modality per call."""
    B = xs[0].shape[0]
    F = int(mask.max()) + 1
    P, Fp = perms.shape
    ranks = torch.full((P, F), Fp, dtype=torch.long, device=mask.device)
    for p in range(P):
        ranks[p, perms[p].to(mask.device)] = torch.arange(Fp, device=mask.device)
    steps = [(p, k) for p in range(P) for k in range(-1, Fp)]
    out = []
    with torch.no_grad():
        for t in range(len(xs)):
            f = []
            for i in range(0, len(steps), chunk):
                part = steps[i:i + chunk]
                sel = torch.cat([(ranks[p][mask] > k).expand(B, -1, -1, -1, -1) for p, k in part])
                comp = xs[t].repeat(len(part), 1, 1, 1, 1).masked_fill_(sel, baseline)
                X = [comp if u == t else x.repeat(len(part), 1, 1, 1, 1) for u, x in enumerate(xs)]
                f.append(model(*X)[0].gather(1, target.repeat(len(part)).view(-1, 1)).view(len(part), B))
            f = torch.cat(f).view(P, Fp + 1, B)
            sc = torch.zeros((B, F), device=mask.device)
            for p in range(P):
                sc[:, perms[p].to(mask.device)] += (f[p, 1:] - f[p, :-1]).t()
            out.append(sc / P)
    return out


def state_bytes(spec, B, P, towers=2):
    """Chain state of one call from the shapes: per chain, sample and tower the bf16 inputs of layers 1-6 and the fp32 tower
    output (floor-mode pooling)."""
    ext, per = [SHAPE], 0
    for _, _, _, pool in spec.layers:
        ext.append(tuple(e // 2 for e in ext[-1]) if pool != L.POOL_NONE else ext[-1])
    for l, (cin, _, _, _) in enumerate(spec.layers):
        if l > 0:
            per += int(np.prod(ext[l])) * cin * 2
    per += int(np.prod(ext[-1])) * spec.layers[-1][1] * 4
    return {"per_chain_sample_tower": per, "total": per * B * P * towers}


def run(B, cells, P, ibs):
    model, mri, pet, label = model_ad(B)
    model.eval().requires_grad_(False)
    xs = [mri, pet]
    spec = model.mri_cnn._spec
    mask = make_atlas(SHAPE, cells, seed=0).cuda()
    chunk = max(1, ibs // B)

    def inc():
        torch.manual_seed(0)
        return shapley_sampling(model, xs, label, mask, 0.0, n_samples=P, internal_batch_size=ibs)

    res = inc()
    perms = res.permutations
    brute = lambda: brute_force(model, xs, label, mask, perms, 0.0, chunk)
    ref = brute()
    with torch.no_grad():
        fx = model(*xs)[0].gather(1, label.view(-1, 1)).view(-1)
    scale = float(fx.abs().max())
    err = max(float((a - b).abs().max()) for a, b in zip(res.scores, ref))
    out = {"players": int(perms.shape[1]), "n_samples": P, "chains_per_pass_cap": chunk, "incremental_ms": [],
           "brute_force_ms": [], "max_abs_score_diff_over_max_abs_fx": round(err / scale, 6),
           "max_abs_delta_over_max_abs_fx": round(max(float(d.abs().max()) for d in res.delta) / scale, 6)}
    for _ in range(3):                         # alternate: drift of the shared host hits both
        out["incremental_ms"].append(round(timed(inc, 1, warmup=1), 1))
        out["brute_force_ms"].append(round(timed(brute, 1, warmup=0), 1))
    f, p = min(out["incremental_ms"]), min(out["brute_force_ms"])
    out.update(incremental_subjects_per_s=round(B / f * 1e3, 3), brute_force_subjects_per_s=round(B / p * 1e3, 3),
               speedup=round(p / f, 3), target_speedup=3.0, target_met=p / f >= 3.0)
    # the schedule the call ran, from the permutations alone
    boxes = TF.abl_boxes(mask, int(mask.max()) + 1)
    classes = TF.abl_classes(boxes, SHAPE)
    layers = [(ks, pool) for _, _, ks, pool in spec.layers]
    caps = [min(chunk, TF.occ_pass_limit(TF.abl_plan(boxes, ids, SHAPE, layers), spec, B, 2)) for _, ids in classes]
    cls_of = {fid: c for c, (_, ids) in enumerate(classes) for fid in ids}
    passes = len(TF.shap_schedule(perms.numpy(), cls_of, caps))
    out.update(passes=passes, mean_chains_per_pass=round(perms.numel() / passes, 2), state_bytes=state_bytes(spec, B, P))
    # host time to enqueue one call (it returns before the device finishes) against its wall time
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    inc()
    t1 = time.perf_counter()
    torch.cuda.synchronize()
    t2 = time.perf_counter()
    # one call under per-launch events: crop launches against the rest (two base forwards and f(start) once, the fusion
    # stack per pass)
    L.TIMER.start()
    inc()
    rec = L.TIMER.stop()
    L.TIMER.start()
    with torch.no_grad():
        model(*xs)
    base = sum(ms for ms, _ in L.TIMER.stop().values())
    crop = lambda tag: ("occ" in tag or "shap" in tag)
    tower = sum(ms for tag, (ms, _) in rec.items() if crop(tag))
    rest = sum(ms for tag, (ms, _) in rec.items() if not crop(tag) and tag != "tmf_abl_map")
    out["per_pass_ms"] = {"crop_launches": round(tower / passes, 3),
                          "fusion_plus_heads": round((rest - 2 * base) / passes, 3),
                          "host_enqueue": round((t1 - t0) * 1e3 / passes, 3),
                          "wall": round((t2 - t0) * 1e3 / passes, 3)}
    out["call_host_enqueue_ms"], out["call_wall_ms"] = round((t1 - t0) * 1e3, 1), round((t2 - t0) * 1e3, 1)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--cells", type=int, default=96)
    ap.add_argument("--samples", type=int, default=25)
    ap.add_argument("--internal-batch", type=int, default=256)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("shapley_bench.py measures on the GPU; no CUDA device found")
    res = {"gpu": gpu_info(), "torch_device": torch.cuda.get_device_name(), "shape": SHAPE, "model": "model_ad eval",
           "headline": {"batch": a.batch, "cells": a.cells, "internal_batch_size": a.internal_batch,
                        **run(a.batch, a.cells, a.samples, a.internal_batch)}}
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
