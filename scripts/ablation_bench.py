"""Feature-ablation measurements on one GPU, in one process:

  1. interpret.feature_ablation(model_ad) over a seeded synthetic atlas (incremental: each region recomputes only what its
     bounding box changes) against the brute-force loop a user writes by hand (one model call per pass on materialised
     ablated volumes, one modality at a time), with the same regions and the same volumes per pass, alternated three times:
     ms per call and subjects/s;
  2. the same for each candidate extent-class ladder (``functional.ABL_LADDER``), alternated with the default;
  3. one incremental call under per-launch CUDA events: the tower part (crop launches) and the fusion-plus-heads part per
     pass;
  4. the conv work the crops launch against brute force's, computed from the shapes;
  5. the GPU name and power limit, read in the same run (nvidia-smi query only).

Usage: python scripts/ablation_bench.py [--batch 8] [--cells 96] [--internal-batch 256] [--out FILE]
Defaults: model_ad in eval mode, B = 8 subjects of 91 x 109 x 91, 96 Voronoi cells plus background, baseline 0.  A brute-force
pass moves gigabytes, far beyond the 126 MB L2.
"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from saliency_bench import SHAPE, gpu_info, model_ad, timed   # noqa: E402
from transmf_ad_b200 import _lib as L                         # noqa: E402
from transmf_ad_b200 import functional as TF                  # noqa: E402
from transmf_ad_b200.interpret import feature_ablation        # noqa: E402
from transmf_ad_b200.synthetic import make_atlas              # noqa: E402

# candidate extent-class ladders: fine (~1.5x rungs), medium, coarse (powers of two)
LADDERS = {"x1.5": (8, 12, 16, 24, 32, 48, 64, 96, 128), "x2_from24": (24, 48, 96), "x2": (16, 32, 64, 128)}


def brute_force(model, xs, target, mask, ids, baseline, chunk):
    """Scores from the model's own forward on materialised ablated volumes, ``chunk`` regions of one modality per call."""
    B = xs[0].shape[0]
    out = []
    with torch.no_grad():
        fx = model(*xs)[0].gather(1, target.view(-1, 1)).view(-1)
        for t in range(len(xs)):
            sc = []
            for k0 in range(0, len(ids), chunk):
                part = ids[k0:k0 + chunk]
                sel = torch.cat([(mask == f).expand(B, -1, -1, -1, -1) for f in part])
                abl = xs[t].repeat(len(part), 1, 1, 1, 1).masked_fill_(sel, baseline)
                X = [abl if u == t else x.repeat(len(part), 1, 1, 1, 1) for u, x in enumerate(xs)]
                sc.append(fx.view(1, B) - model(*X)[0].gather(1, target.repeat(len(part)).view(-1, 1)).view(len(part), B))
            out.append(torch.cat(sc))
    return out


def conv_work(boxes, spec, B, towers=2):
    """Conv FLOPs per call from the shapes: the incremental crops of every extent class against brute force (every region,
    both towers of the model call run in full, one modality ablated per call)."""
    layers = [(ks, pool) for _, _, ks, pool in spec.layers]
    classes = TF.abl_classes(boxes, SHAPE)
    inc = full = 0
    for _, ids in classes:
        plan = TF.abl_plan(boxes, ids, SHAPE, layers)
        for l, (cin, cout, ks, pool) in enumerate(spec.layers):
            f = 2 * cin * cout * ks ** 3
            inc += towers * plan.n * B * plan.crop[l][0] * plan.crop[l][1] * plan.crop[l][2] * f
            full += towers * towers * plan.n * B * plan.full[l][0] * plan.full[l][1] * plan.full[l][2] * f
    # the same regions, each on a crop planned for its own box alone (no padding to a class extent)
    own = 0
    for _, ids in classes:
        for fid in ids:
            plan = TF.abl_plan(boxes, [fid], SHAPE, layers)
            for l, (cin, cout, ks, pool) in enumerate(spec.layers):
                own += towers * B * plan.crop[l][0] * plan.crop[l][1] * plan.crop[l][2] * 2 * cin * cout * ks ** 3
    return {"classes": len(classes), "regions_per_class": [len(ids) for _, ids in classes],
            "incremental_gflop": round(inc / 1e9, 1), "brute_force_gflop": round(full / 1e9, 1),
            "ratio": round(inc / full, 4), "ratio_without_class_padding": round(own / full, 4)}


def run(B, cells, ibs):
    model, mri, pet, label = model_ad(B)
    model.eval().requires_grad_(False)
    xs = [mri, pet]
    spec = model.mri_cnn._spec
    mask = make_atlas(SHAPE, cells, seed=0).cuda()
    F = int(mask.max()) + 1
    boxes = TF.abl_boxes(mask, F)
    ids = [f for f in range(F) if boxes[f, 3] > boxes[f, 0]]
    chunk = max(1, ibs // B)
    inc = lambda: feature_ablation(model, xs, label, mask, 0.0, internal_batch_size=ibs)
    brute = lambda: brute_force(model, xs, label, mask, ids, 0.0, chunk)
    default = TF.ABL_LADDER
    a, b = inc().scores, brute()
    err = [float((x[:, ids].t() - y).abs().max()) for x, y in zip(a, b)]
    with torch.no_grad():
        fx = model(*xs)[0].gather(1, label.view(-1, 1)).view(-1)
    out = {"regions": len(ids), "regions_per_pass": chunk, "ladder": list(default), "incremental_ms": [],
           "brute_force_ms": [], "max_abs_score_diff_over_max_abs_fx": round(max(err) / float(fx.abs().max()), 6)}
    for _ in range(3):                         # alternate: drift of the shared host hits both
        out["incremental_ms"].append(round(timed(inc, 1, warmup=1), 1))
        out["brute_force_ms"].append(round(timed(brute, 1, warmup=0), 1))
    f, p = min(out["incremental_ms"]), min(out["brute_force_ms"])
    out.update(incremental_subjects_per_s=round(B / f * 1e3, 3), brute_force_subjects_per_s=round(B / p * 1e3, 3),
               speedup=round(p / f, 3), target_speedup=3.0, target_met=p / f >= 3.0)
    # the extent-class ladder: every candidate alternated with the default in the same run
    lad = {}
    for name, ladder in LADDERS.items():
        ms = []
        for _ in range(3):
            TF.ABL_LADDER = ladder
            ms.append(round(timed(inc, 1, warmup=1), 1))
            TF.ABL_LADDER = default
            ms.append(round(timed(inc, 1, warmup=1), 1))
        TF.ABL_LADDER = ladder
        lad[name] = {"ladder": list(ladder), "ms": ms[0::2], "default_ms": ms[1::2], "conv_work": conv_work(boxes, spec, B)}
        TF.ABL_LADDER = default
    out["ladders"] = lad
    # one call under per-launch events: crop launches against the rest (the base forward once, the fusion stack per pass)
    passes = sum(-(-len(c) // chunk) for _, c in TF.abl_classes(boxes, SHAPE))
    L.TIMER.start()
    inc()
    rec = L.TIMER.stop()
    L.TIMER.start()
    with torch.no_grad():
        model(*xs)
    base = sum(ms for ms, _ in L.TIMER.stop().values())
    crop = lambda tag: ("occ" in tag or "abl_input" in tag)
    tower = sum(ms for tag, (ms, _) in rec.items() if crop(tag))
    rest = sum(ms for tag, (ms, _) in rec.items() if not crop(tag) and tag != "tmf_abl_map")
    out["passes"] = passes
    out["kernel_time_per_pass_ms"] = {"tower_part": round(tower / passes, 2),
                                      "fusion_plus_heads": round((rest - base) / passes, 2),
                                      "base_forward_once": round(base, 2),
                                      "abl_map_once": round(rec.get("tmf_abl_map", (0.0, 0))[0], 3)}
    out["conv_work"] = conv_work(boxes, spec, B)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--cells", type=int, default=96)
    ap.add_argument("--internal-batch", type=int, default=256)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ablation_bench.py measures on the GPU; no CUDA device found")
    res = {"gpu": gpu_info(), "torch_device": torch.cuda.get_device_name(), "shape": SHAPE, "model": "model_ad eval",
           "headline": {"batch": a.batch, "cells": a.cells, "internal_batch_size": a.internal_batch,
                        **run(a.batch, a.cells, a.internal_batch)}}
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
