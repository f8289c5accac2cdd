"""Occlusion-sensitivity measurements on one GPU, in one process:

  1. interpret.occlusion(model_ad) (incremental: only the region each window changes is recomputed) against the brute-force
     loop a user writes by hand (one model call per pass on materialised occluded volumes, one modality at a time), with the
     same windows and the same volumes per pass, alternated three times: ms per batch and subjects/s;
  2. one incremental call under per-launch CUDA events: the tower part (crop launches, tagged ``@occ``) and the
     fusion-plus-heads part per pass, and the per-call time and bytes/s of the compose kernels;
  3. the conv work the crops launch against brute force's, computed from the shapes, and which conv kernel each crop
     layer takes (tcgen05 column / tcgen05 streamed / direct);
  4. the GPU name and power limit, read in the same run (nvidia-smi query only).

Usage: python scripts/occlusion_bench.py [--batch 8] [--window 16] [--stride 16] [--internal-batch 256] [--out FILE]
Defaults: the headline configuration, model_ad in eval mode, B = 8 subjects of 91 x 109 x 91.  A brute-force pass moves
gigabytes, far beyond the 126 MB L2.
"""
import argparse
import ctypes
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from saliency_bench import COPY_PEAK, SHAPE, gpu_info, model_ad, timed   # noqa: E402
from transmf_ad_b200 import _lib as L                                    # noqa: E402
from transmf_ad_b200 import functional as TF                             # noqa: E402
from transmf_ad_b200.interpret import occlusion                          # noqa: E402


def brute_force(model, xs, target, window, stride, baseline, chunk):
    """Scores from the model's own forward on materialised occluded volumes, ``chunk`` windows of one modality per call."""
    B = xs[0].shape[0]
    starts = [TF.occ_positions(E, w, s) for E, w, s in zip(SHAPE, window, stride)]
    wins = [(a, b, c) for a in starts[0] for b in starts[1] for c in starts[2]]
    out = []
    with torch.no_grad():
        fx = model(*xs)[0].gather(1, target.view(-1, 1)).view(-1)
        for t in range(len(xs)):
            sc = []
            for k0 in range(0, len(wins), chunk):
                part = wins[k0:k0 + chunk]
                occ = xs[t].repeat(len(part), 1, 1, 1, 1)
                for n, (a, b, c) in enumerate(part):
                    occ[n * B:(n + 1) * B, :, a:a + window[0], b:b + window[1], c:c + window[2]] = baseline
                X = [occ if u == t else x.repeat(len(part), 1, 1, 1, 1) for u, x in enumerate(xs)]
                sc.append(fx.view(1, B) - model(*X)[0].gather(1, target.repeat(len(part)).view(-1, 1)).view(len(part), B))
            out.append(torch.cat(sc))
    return out


def conv_work(plan, spec, m, B, passes, nwin, towers=2):
    """Conv FLOPs per call from the shapes: the incremental crops (all passes) against brute force (every window, both
    towers of the model call run in full, one modality occluded per call), and the kernel each crop layer takes."""
    inc = full = 0
    kern = []
    for l, (cin, cout, ks, pool) in enumerate(spec.layers):
        Dc, Hc, Wc = plan.crop[l]
        D, H, W = plan.full[l]
        f = 2 * cin * cout * ks ** 3
        inc += towers * nwin * B * Dc * Hc * Wc * f
        full += towers * towers * nwin * B * D * H * W * f
        if l == 0:
            kern.append("tcgen05 conv1" if cout in (32, 64) else "direct")
            continue
        info = (ctypes.c_int * 6)()
        if not L.load().tmf_conv3d_supported(0, L.CONV_UMMA, Dc, Hc, Wc, cin, cout, ks):
            kern.append("direct")
        elif L.load().tmf_conv3d_col_plan_info(towers, Dc, Hc, Wc, cin, cout, ks, info) == 0:
            kern.append("tcgen05 column")
        else:
            kern.append("tcgen05 streamed")
    return {"incremental_gflop": round(inc / 1e9, 1), "brute_force_gflop": round(full / 1e9, 1),
            "ratio": round(inc / full, 4), "crop_extents": plan.crop[:7], "crop_kernels": kern}


def run(B, window, stride, ibs):
    model, mri, pet, label = model_ad(B)
    model.eval().requires_grad_(False)
    xs = [mri, pet]
    window, stride = (window,) * 3, (stride,) * 3
    spec = model.mri_cnn._spec
    plan = TF.OccPlan(SHAPE, window, stride, [(ks, pool) for _, _, ks, pool in spec.layers])
    chunk = max(1, ibs // B)
    passes = -(-plan.nwin // chunk)
    inc = lambda: occlusion(model, xs, label, window=window, stride=stride, internal_batch_size=ibs)
    brute = lambda: brute_force(model, xs, label, window, stride, 0.0, chunk)
    a, b = inc().scores, brute()
    err = [float((x.reshape(B, -1).t() - y).abs().max()) for x, y in zip(a, b)]
    with torch.no_grad():
        fx = model(*xs)[0].gather(1, label.view(-1, 1)).view(-1)
    out = {"windows_per_tower": plan.nwin, "windows_per_pass": chunk, "passes": passes, "incremental_ms": [],
           "brute_force_ms": [], "max_abs_score_diff_over_max_abs_fx": round(max(err) / float(fx.abs().max()), 5)}
    for _ in range(3):                         # alternate: drift of the shared host hits both
        out["incremental_ms"].append(round(timed(inc, 1, warmup=1), 1))
        out["brute_force_ms"].append(round(timed(brute, 1, warmup=0), 1))
    f, p = min(out["incremental_ms"]), min(out["brute_force_ms"])
    out.update(incremental_subjects_per_s=round(B / f * 1e3, 3), brute_force_subjects_per_s=round(B / p * 1e3, 3),
               speedup=round(p / f, 3), target_speedup=3.0, target_met=p / f >= 3.0)
    # one call under per-launch events: crop launches against the rest (the base forward once, the fusion stack per pass)
    L.TIMER.start()
    inc()
    rec = L.TIMER.stop()
    L.TIMER.start()
    with torch.no_grad():
        model(*xs)
    base = sum(ms for ms, _ in L.TIMER.stop().values())
    tower = sum(ms for tag, (ms, _) in rec.items() if "occ" in tag)
    rest = sum(ms for tag, (ms, _) in rec.items() if "occ" not in tag)
    out["kernel_time_per_pass_ms"] = {"tower_part": round(tower / passes, 2),
                                      "fusion_plus_heads": round((rest - base) / passes, 2),
                                      "base_forward_once": round(base, 2)}
    comp = {}
    for tag, (ms, n) in sorted(rec.items()):
        if not tag.startswith("tmf_occ_compose"):
            continue
        where = tag.split("@")[1]
        if where.startswith("L"):
            l = int(where[1:])
            elems = chunk * B * plan.crop[l][0] * plan.crop[l][1] * plan.crop[l][2] * spec.layers[l][0] * 2 * 2
        else:                                  # fp32 tower outputs, both towers of a pass
            elems = chunk * B * plan.crop[7][0] * plan.crop[7][1] * plan.crop[7][2] * spec.dim * 4 * 2
        nbytes = 2 * elems                     # every output byte read once from one source and written once
        comp[tag] = {"ms_per_call": round(ms / n, 4), "calls": n, "bytes_per_call": nbytes,
                     "GB_per_s": round(nbytes / (ms / n) / 1e6, 1),
                     "fraction_of_copy_peak": round(nbytes / (ms / n * 1e-3) / COPY_PEAK, 3)}
    out["compose_kernels"] = comp
    out["conv_work"] = conv_work(plan, spec, chunk, B, passes, plan.nwin)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--window", type=int, default=16)
    ap.add_argument("--stride", type=int, default=16)
    ap.add_argument("--internal-batch", type=int, default=256)
    ap.add_argument("--also-stride8-b2", action="store_true", help="add the stride-8 configuration at B = 2")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("occlusion_bench.py measures on the GPU; no CUDA device found")
    res = {"gpu": gpu_info(), "torch_device": torch.cuda.get_device_name(), "shape": SHAPE, "model": "model_ad eval",
           "headline": {"batch": a.batch, "window": a.window, "stride": a.stride, "internal_batch_size": a.internal_batch,
                        **run(a.batch, a.window, a.stride, a.internal_batch)}}
    if a.also_stride8_b2:
        res["stride8_b2"] = {"batch": 2, "window": a.window, "stride": 8, "internal_batch_size": a.internal_batch,
                             **run(2, a.window, 8, a.internal_batch)}
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
