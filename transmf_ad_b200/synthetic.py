"""Deterministic synthetic MRI/PET volumes and procedural weights shared by bench.py and the tests.

The reference feeds each model fp32 volumes of shape (B,1,D,H,W) scaled to [0,1] by MONAI's
``ScaleIntensityd`` (reference datasets/ADNI.py:59-84; native size, no crop / pad).  There is no dataset in
this environment, so volumes are synthesised on the CPU generator (bit-reproducible for a given torch build):
a smooth low-resolution random field, tri-linearly up-sampled, plus voxel noise and a class-dependent blob
(pure i.i.d. noise would make all subjects nearly identical after the CNN and degenerate the BatchNorm1d
heads -- SURVEY.md section 8d).
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

PRIMARY_SHAPE = (91, 109, 91)        # MNI152 2 mm grid, reference datasets/ADNI.py:93


def make_volumes(batch, shape=PRIMARY_SHAPE, seed=1, labels=None, device="cpu"):
    """-> (B,1,D,H,W) fp32 in [0,1].  ``labels`` (B,) int adds a class-dependent blob."""
    g = torch.Generator().manual_seed(int(seed))
    D, H, W = shape
    low = torch.rand(batch, 1, 12, 14, 12, generator=g)
    vol = F.interpolate(low, size=(D, H, W), mode="trilinear", align_corners=False)
    vol = vol + 0.05 * torch.rand(batch, 1, D, H, W, generator=g)
    if labels is None:
        labels = torch.arange(batch) % 2
    zz = torch.linspace(-1, 1, D).view(D, 1, 1)
    yy = torch.linspace(-1, 1, H).view(1, H, 1)
    xx = torch.linspace(-1, 1, W).view(1, 1, W)
    for b in range(batch):
        c = 0.35 if int(labels[b]) else -0.35
        blob = torch.exp(-(((zz - c) ** 2 + (yy + c) ** 2 + xx ** 2) / 0.08))
        vol[b, 0] += 0.6 * blob
    lo = vol.amin(dim=(1, 2, 3, 4), keepdim=True)
    hi = vol.amax(dim=(1, 2, 3, 4), keepdim=True)
    vol = (vol - lo) / (hi - lo)                      # per-volume min-max, like ScaleIntensityd
    return vol.contiguous().to(device)


def make_atlas(shape=PRIMARY_SHAPE, cells=96, seed=0, radius=0.42):
    """-> int64 (1,1,D,H,W) synthetic parcellation: ``cells`` Voronoi cells (ids 1 .. cells) of seeded centres inside an
    ellipsoid of semi-axes ``radius`` times the extent, background 0 outside it (a stand-in for an anatomical atlas)."""
    g = torch.Generator().manual_seed(int(seed))
    D, H, W = shape
    grid = torch.stack(torch.meshgrid(torch.arange(D), torch.arange(H), torch.arange(W), indexing="ij"), -1).reshape(-1, 3)
    grid = grid.double()
    centre = torch.tensor([(D - 1) / 2, (H - 1) / 2, (W - 1) / 2], dtype=torch.float64)
    semi = radius * torch.tensor([D, H, W], dtype=torch.float64)
    inside = (((grid - centre) / semi) ** 2).sum(1) <= 1
    pts = grid[inside]
    seeds = pts[torch.randperm(len(pts), generator=g)[:cells]]
    lab = torch.zeros(D * H * W, dtype=torch.int64)
    cell = torch.cat([torch.cdist(pts[i:i + 65536], seeds).argmin(1) for i in range(0, len(pts), 65536)])
    lab[inside] = cell + 1
    return lab.view(1, 1, D, H, W)


def make_labels(batch, device="cpu"):
    return (torch.arange(batch) % 2).to(torch.int64).to(device)


def procedural_state(template, seed=0):
    """Fill a state-dict *template* (key -> tensor giving shape/dtype) with deterministic values.

    Values are drawn per key, in the template's own key order, from a CPU generator, with scales that mimic
    the reference initialisation (kaiming fan_out for conv, 1/sqrt(fan_in) for linear, reference
    models/mymodel.py:195-202) but with non-trivial BN/LN affine parameters and running statistics so that
    every term of every formula is exercised."""
    g = torch.Generator().manual_seed(int(seed))
    out = {}
    for k, t in template.items():
        shape = tuple(t.shape)
        if k.endswith("num_batches_tracked"):
            v = torch.zeros(shape, dtype=torch.int64)
        elif k.endswith("running_mean"):
            v = 0.1 * torch.randn(shape, generator=g)
        elif k.endswith("running_var"):
            v = 1.0 + 0.2 * torch.rand(shape, generator=g)
        elif len(shape) == 5:                          # Conv3d weight (Cout,Cin,kd,kh,kw)
            fan_out = shape[0] * shape[2] * shape[3] * shape[4]
            v = torch.randn(shape, generator=g) * (2.0 / fan_out) ** 0.5
        elif len(shape) == 2:                          # Linear weight (out,in)
            bound = 1.0 / shape[1] ** 0.5
            v = (torch.rand(shape, generator=g) * 2 - 1) * bound
        elif k.endswith("weight"):                     # BN / LN scale
            v = 1.0 + 0.1 * torch.randn(shape, generator=g)
        else:                                          # biases / shifts
            v = 0.05 * torch.randn(shape, generator=g)
        out[k] = v.to(t.dtype) if t.is_floating_point() else v
    return out
