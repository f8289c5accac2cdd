#!/usr/bin/env python
"""bench.py -- train subjects/s (MRI+PET pairs) of the TransMF_AD hot path on B200.

    python bench.py --gpus N --steps K --warmup W [--workload both|ad|cnn_ad|single] [--batch B] [--impl reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

One "step" = the caller's train_step (reference kfold_train_adversarial.py:101-136): forward, CE + adversarial
losses, backward, (gradient all-reduce for N > 1) and the Adam step of utils/utils.py:38-41, on one batch of
synthetic paired volumes of shape (B,1,91,109,91).  Rank 0 prints ONE JSON line.

Headline (``value``, ``e2e``, ``roofline``): BASELINE configs[2] = ``model_ad`` (``--model Transformer``, the reference's
main entry), batch 8 per GPU, weak scaling.  ``workloads`` carries the same numbers for configs[1] (``model_CNN_ad``,
``--model CNN``) beside it.

``value``         device-timed (CUDA events, max over ranks) with the batch already resident in HBM.
``e2e``           same step driven from PINNED HOST buffers: H2D copy of MRI/PET/labels and the two loss reads (D2H) inside
                  the timed region.
``roofline``      conv3d kernels conv2.0 .. conv4.3 (fwd + dgrad + wgrad, algorithmic FLOPs of SURVEY.md section 8d): CUDA events
                  around every launch of one step whose launches were enqueued behind a spin kernel (so the events see
                  back-to-back device execution, not host launch gaps), against the measured BURST bf16 peak (kernels of
                  20-230 us timed one by one run at full clock); the sustained-peak fraction is given beside it.
``eager_dropin``  what the UNCHANGED reference loop gets: eager launches + torch.optim.Adam + .item() reads, host buffers.
``sustained``     >= 2000 graph replays back to back with the clock record (steady-state clocks / power).
``c4``            (N > 1) BASELINE configs[3]: model_ad, global batch 64 split over the ranks (strong scaling).
``cpu_baseline``  the CPU oracle port (oracle/restatement.py; the reference is pure PyTorch) timed on the host cores on
                  BASELINE configs[0] (model_ad, batch 2).
``--impl reference`` times that CPU port alone (batch 2 per step -- stated in config.workload -- honouring --steps/--warmup)
                  and prints the same line shape with "impl": "reference".
``--dump-outputs DIR`` writes what the last timed step of each measured workload computed -- the losses and model outputs
                  it returns and the parameters, gradients and buffers it updates in place -- as DIR/<workload>.<name>.npy
                  (float32, or float64 for integer buffers).  Inputs, weights and dropout masks are seeded, so two builds
                  run with the same arguments can be compared array for array.
"""
from __future__ import annotations

import argparse
import gc
import hashlib
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SHAPE = (91, 109, 91)
METRIC = "train subjects/s (MRI+PET pairs)"
WORKLOADS = {
    # name: (model class, ctor kwargs, towers, description)
    "cnn_ad": ("model_CNN_ad", dict(dim=128), 2, "model_CNN_ad (--model CNN) adversarial train step"),
    "ad": ("model_ad", dict(dim=128, depth=3, heads=4, dim_head=32, mlp_dim=512, dropout=0.), 2,
           "model_ad (--model Transformer) adversarial train step"),
    "single": ("model_single", dict(dim=128), 1, "model_single (kfold_train_single) train step"),
    # BASELINE configs[4] (MiSePyNet baseline, kfold_train_Mnet.py:85: SGD lr 1e-3 momentum 0.9, CE loss); not the headline
    "mnet": ("Mnet", dict(), 2, "Mnet / MiSePyNet baseline (kfold_train_Mnet.py) train step"),
}
CPU_SAMPLE_BATCH = 2      # BASELINE configs[0] / the reference's default --batch_size
OUTPUT_NAMES = ("logits", "d_mri_logits", "d_pet_logits")      # model_ad / model_CNN_ad return all three, the others logits
LOSS_NAMES = ("loss_total", "loss_ce", "loss_ad")
DUMP_BYTES = 64 * 10 ** 6                                      # --dump-outputs: all .npy files together stay below this


def conv_flops_per_subject(shape, dim=128, towers=2, first_layer=True, other_layers=True):
    """Algorithmic conv FLOPs: 2*M*Cout*Cin*k^3 for fwd and wgrad of every layer and dgrad of all but conv1.0.
    ``first_layer`` / ``other_layers`` select conv1.0 (Cin = 1, HBM-bound) and conv2.0 .. conv4.3 (tensor-bound)."""
    from transmf_ad_b200.functional import SNetSpec
    D, H, W = shape
    total = 0.0
    for l, (cin, cout, ks, pool) in enumerate(SNetSpec(dim).layers):
        f = 2.0 * D * H * W * cout * cin * ks ** 3
        if (l == 0 and first_layer) or (l > 0 and other_layers):
            total += f * (3 if l > 0 else 2)
        if pool:
            D, H, W = D // 2, H // 2, W // 2
    return total * towers


def block1_bytes_per_subject(shape, dim=128, towers=2):
    """Algorithmic HBM bytes of the four block-1 passes (SURVEY.md section 8d): x fp32, y bf16 (dim/4 channels),
    pooled activation / its gradient bf16."""
    D, H, W = shape
    c = dim // 4
    x = 4.0 * D * H * W
    y = 2.0 * D * H * W * c
    pooled = 2.0 * (D // 2) * (H // 2) * (W // 2) * c
    from transmf_ad_b200.functional import keep_ymax
    keep = keep_ymax()           # forward also writes ymax (pooled extent); the backward reduction reads ymax + dout only
    return {"tmf_conv1_fwd": towers * (x + y), "tmf_bn_act_pool_fwd@L0": towers * (y + pooled * (2 if keep else 1)),
            "tmf_bn_act_pool_bwd_reduce@L0": towers * ((2 * pooled) if keep else (y + pooled)),
            "tmf_conv1_bwd_fused": towers * (y + pooled + x)}


def committed_traffic():
    """DRAM bytes per step of the tensor-bound conv launches from the committed `ncu --set full` capture
    (profiles/conv_traffic.json, written by scripts/ncu_traffic.py); None when absent."""
    path = os.path.join(ROOT, "profiles", "conv_traffic.json")
    if not os.path.exists(path):
        return None
    with open(path) as f:
        return json.load(f)


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"],
                "bf16_tflops_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


def library_hash():
    """sha256 (first 16 hex) of the loaded libtmf_sm100a.so and of the sources it was built from (stale-binary check)."""
    from transmf_ad_b200 import _lib, build
    with open(_lib.LIB_PATH, "rb") as f:
        so = hashlib.sha256(f.read()).hexdigest()[:16]
    return {"so_sha256_16": so, "sources_sha256_16": build.source_hash()[:16], "built_from": build.recorded_hash()[:16]}


def step_arrays(model, outs, step_losses):
    """Host copies of what one train step gave its caller: the losses and model outputs it returned, and the parameters,
    gradients and buffers (BatchNorm statistics) it left in the model.  Integer buffers become float64, the rest float32."""
    def host(t):
        t = t.detach()
        return (t.float() if t.is_floating_point() else t.double()).cpu().numpy()

    arrays = {name: host(t) for name, t in zip(LOSS_NAMES, step_losses) if t is not None}
    arrays.update({name: host(t) for name, t in zip(OUTPUT_NAMES, outs)})
    for k, p in model.named_parameters():
        arrays[f"param.{k}"] = host(p)
        if p.grad is not None:
            arrays[f"grad.{k}"] = host(p.grad)
    arrays.update({f"buffer.{k}": host(b) for k, b in model.named_buffers()})
    return arrays


def write_dump(path, arrays):
    """Write ``{name: array}`` as path/<name>.npy.  Past DUMP_BYTES every array keeps the same fraction of its elements,
    at positions (of the flattened array, ascending) drawn from a generator seeded with the array's name: runs with the
    same arguments store the same positions."""
    import zlib
    import numpy as np
    os.makedirs(path, exist_ok=True)
    per_file = 128 + 8                               # .npy header, and the one element a tiny array keeps
    total = sum(a.nbytes for a in arrays.values())
    frac = min(1.0, (DUMP_BYTES - per_file * len(arrays)) / max(total, 1))
    for name, a in arrays.items():
        if frac < 1.0:
            keep = max(1, int(a.size * frac))
            pos = np.random.default_rng(zlib.crc32(name.encode())).choice(a.size, keep, replace=False)
            a = a.reshape(-1)[np.sort(pos)]
        np.save(os.path.join(path, name + ".npy"), a)
    return {"dir": path, "arrays": len(arrays), "sampled": frac < 1.0}


class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.proc = None
        self.index = index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            out, _ = self.proc.communicate()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1])); power.append(float(parts[2]))
            except ValueError:
                continue
            for n, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "power_w_max": max(power),
                "samples": len(sm), "reasons": sorted(reasons)}


def pin_to_local_numa(local_rank, world):
    """CPU affinity of this rank = its share of the cores of the GPU's NUMA node (pinned-buffer pages are then allocated and
    copied from node-local memory; round 1 had every rank on cores 0-31 of node 0: 31 GB/s H2D per rank at N = 8)."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=index,pci.bus_id", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=20).stdout
        node_of = {}
        for line in out.strip().splitlines():
            idx, bus = [x.strip() for x in line.split(",")]
            bus = bus.lower()
            if len(bus.split(":")[0]) == 8:                  # 00000000:1b:00.0 -> 0000:1b:00.0
                bus = bus[4:]
            with open(f"/sys/bus/pci/devices/{bus}/numa_node") as f:
                node_of[int(idx)] = int(f.read().strip())
        visible = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = [int(x) for x in visible.split(",")] if visible and all(x.strip().isdigit() for x in visible.split(",")) \
            else sorted(node_of)
        node = node_of[phys[local_rank]]
        if node < 0:
            return {"numa_node": -1}
        cpus = []
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            for part in f.read().strip().split(","):
                a, _, b = part.partition("-")
                cpus += list(range(int(a), int(b or a) + 1))
        allowed = sorted(set(cpus) & os.sched_getaffinity(0)) or sorted(os.sched_getaffinity(0))
        peers = [r for r in range(world) if r < len(phys) and node_of.get(phys[r]) == node]      # ranks sharing the node
        if local_rank in peers and len(peers) > 1:
            per = max(1, len(allowed) // len(peers))
            i = peers.index(local_rank)
            mine = allowed[i * per:(i + 1) * per] or allowed
        else:
            mine = allowed
        os.sched_setaffinity(0, mine)
        torch.set_num_threads(max(1, min(len(mine), 8)))
        return {"numa_node": node, "cpus": f"{mine[0]}-{mine[-1]} ({len(mine)})"}
    except Exception as e:                                    # affinity is an optimisation, never a failure
        return {"error": str(e)[:120]}


# ------------------------------------------------------------------------------------------------------------------
def cpu_port_step_fn(workload, batch):
    """The CPU oracle port of the same train step (fwd + losses + bwd + Adam) on a bounded sample."""
    from oracle import restatement as R
    from transmf_ad_b200.models import mymodel as M
    from transmf_ad_b200.synthetic import make_labels, make_volumes, procedural_state
    kind, kwargs, towers, _ = WORKLOADS[workload]
    template = getattr(M, kind)(**kwargs).state_dict()
    sd = R.clone_state(procedural_state(template, seed=0))
    label = make_labels(batch)
    mri = make_volumes(batch, SHAPE, seed=1, labels=label)
    pet = make_volumes(batch, SHAPE, seed=2, labels=label)
    params = [v for k, v in sd.items() if v.is_floating_point() and v.requires_grad]
    opt = torch.optim.Adam(params, lr=1e-4, weight_decay=0.0)
    heads = kwargs.get("heads", 4)

    def step():
        opt.zero_grad()
        if kind == "model_ad":
            outs = R.model_ad_forward(sd, mri, pet, heads=heads, training=True)
        elif kind == "model_CNN_ad":
            outs = R.model_cnn_ad_forward(sd, mri, pet, training=True)
        else:
            outs = (R.model_single_forward(sd, mri, training=True),)
        if len(outs) == 3:
            ce, ad, total = R.adversarial_losses(*outs, label)
        else:
            total = torch.nn.functional.cross_entropy(outs[0], label)
        total.backward()
        opt.step()
        return float(total.detach())

    return step


def time_cpu_port(workload, batch, steps, warmup):
    torch.set_num_threads(os.cpu_count() or 1)
    step = cpu_port_step_fn(workload, batch)
    for _ in range(warmup):
        step()
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        step()
        ts.append(time.perf_counter() - t0)
    return batch * len(ts) / sum(ts), sum(ts) / len(ts), batch / min(ts)


def run_reference_arm(args, rank):
    if rank != 0:
        return
    workload = "ad" if args.workload == "both" else args.workload
    kind, kwargs, towers, desc = WORKLOADS[workload]
    steps, warm = max(1, args.steps), max(0, args.warmup)
    sps, mean_s, best = time_cpu_port(workload, CPU_SAMPLE_BATCH, steps, warm)
    cores = torch.get_num_threads()
    line = {
        "impl": "reference", "metric": METRIC, "value": sps, "unit": "subjects/s", "n_gpus": args.gpus, "steps": steps,
        "warmup": warm, "ms_per_step": mean_s * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{desc}, volumes 91x109x91 fp32, Adam lr 1e-4; CPU arm: bounded sample of batch "
                               f"{CPU_SAMPLE_BATCH} per step (the reference's default --batch_size, BASELINE configs[0]); "
                               f"subjects/s does not depend on the batch on the CPU (8.4 s at batch 8 vs 2.2 s at batch 2, "
                               f"BASELINE.md section 2)",
                   "timed_on": "host CPU", "sample_batch": CPU_SAMPLE_BATCH},
        "cpu_baseline": {"value": sps, "unit": "subjects/s", "cores": cores, "kind": "port", "best_step_value": best,
                         "sample": f"{steps} steps (after {warm} warm-up) of batch {CPU_SAMPLE_BATCH}, mean step, fwd+bwd+Adam, fp32, "
                                   f"torch CPU {torch.__version__}; oracle/restatement.py (the reference is pure PyTorch)"},
        "e2e": {"value": sps, "unit": "subjects/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------------
class Job:
    """One process of the job: device, process group, helpers shared by the measurement legs."""

    def __init__(self, args):
        import torch.distributed as dist
        self.args, self.dist = args, dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        self.affinity = pin_to_local_numa(self.local_rank, self.world) if self.world > 1 else None
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=self.dev)
        if self.world != args.gpus and self.rank == 0:
            print(f"[bench] warning: --gpus {args.gpus} but WORLD_SIZE={self.world}", file=sys.stderr)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, ms):
        t = torch.tensor([ms], device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t)

    def timed(self, fn, steps):
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        self.barrier()
        return self.max_over_ranks(e0.elapsed_time(e1))


def measure(job, workload, B, steps, warmup, mode="graph", optimizer="fused", want_e2e=True, want_roofline=False,
            sustained_steps=0, sample_clocks=False, dump=False):
    """All legs for one workload at per-GPU batch B.  Returns a dict (rank 0 fills the clock record; with ``dump``, rank 0
    adds ``step_arrays`` of the last timed step under "dump")."""
    from transmf_ad_b200 import _lib
    from transmf_ad_b200.dp import FlatGradReducer
    from transmf_ad_b200.models import mymodel as M
    from transmf_ad_b200.synthetic import make_labels, make_volumes, procedural_state
    rank, world, dev = job.rank, job.world, job.dev
    kind, kwargs, towers, desc = WORKLOADS[workload]
    torch.manual_seed(0)                                                     # dropout masks: the same in every run
    if kind == "Mnet":
        from transmf_ad_b200.models.MiSePyNet import Mnet
        model = Mnet()
    else:
        model = getattr(M, kind)(**kwargs)
    model.load_state_dict(procedural_state(model.state_dict(), seed=0))     # identical replicas on every rank
    model = model.to(dev).train()
    graph_mode = mode == "graph"
    if kind == "Mnet":                                                       # kfold_train_Mnet.py:85
        opt = torch.optim.SGD(model.parameters(), lr=1e-3, momentum=0.9)
    elif optimizer == "fused":                                                 # utils/utils.py:38-41 (Adam branch), one launch
        from transmf_ad_b200.optim import FusedAdam
        opt = FusedAdam(model.parameters(), lr=1e-4, weight_decay=0.0)
    else:
        opt = torch.optim.Adam(model.parameters(), lr=1e-4, weight_decay=0.0, capturable=graph_mode)
    reducer = FlatGradReducer(model=model)
    if world > 1:
        reducer.install()
    ce_fn = torch.nn.CrossEntropyLoss()
    ones = torch.ones(B, dtype=torch.int64, device=dev)
    zeros = torch.zeros(B, dtype=torch.int64, device=dev)

    # synthetic batches: a small pool, distinct per rank (seed offsets as in SURVEY.md section 8d)
    npool = 2
    label_h = make_labels(B)
    pool_h = []
    for i in range(npool):
        mri = make_volumes(B, SHAPE, seed=1 + 1000 * rank + i, labels=label_h).pin_memory()
        pet = make_volumes(B, SHAPE, seed=2 + 1000 * rank + i, labels=label_h).pin_memory()
        pool_h.append((mri, pet, label_h.pin_memory()))
    pool_d = [tuple(t.to(dev) for t in b) for b in pool_h]

    def losses(outs, label):
        if len(outs) == 3:                                    # kfold_train_adversarial.py:119-131
            ce = ce_fn(outs[0], label)
            ad = (ce_fn(outs[1], ones) + ce_fn(outs[2], zeros)) / 2
            return ce, ad, ad + ce
        ce = ce_fn(outs[0], label)                           # kfold_train_single.py:105
        return ce, None, ce

    last = {}                                                # eager mode with dump: what the latest step returned

    def train_step(batch, read_losses):                      # the reference's eager loop
        mri, pet, label = batch
        opt.zero_grad()
        outs = model(mri) if towers == 1 else model(mri, pet)
        outs = outs if isinstance(outs, tuple) else (outs,)
        ce, ad, total = losses(outs, label)
        if dump:                                             # detached: a kept autograd graph breaks the graph capture
            last["outs"] = tuple(o.detach() for o in outs)
            last["losses"] = tuple(None if t is None else t.detach() for t in (total, ce, ad))
        vals = None
        if read_losses:                                      # the reference's two .item() syncs (:127-128)
            vals = (ce.item(), ad.item() if ad is not None else 0.0)
        total.backward()
        reducer.finish()
        opt.step()
        return vals

    def inputs_of(batch):
        return batch[:1] if towers == 1 else batch[:2]

    graphed = None
    if graph_mode:
        from transmf_ad_b200.train import DevicePrefetcher, GraphedTrainStep, LossReader

        def graph_loss(outs, label):                         # (total, ce, ad): total.backward() is captured
            ce, ad, total = losses(outs, label)
            return (total, ce) if ad is None else (total, ce, ad)

        for i in range(2):                                   # eager warm-up (lazy inits, allocator, attribute calls)
            train_step(pool_d[i % npool], False)
        job.barrier()
        graphed = GraphedTrainStep(model, opt, graph_loss, inputs_of(pool_d[0]), pool_d[0][2], reducer=reducer, warmup=3)

        def dev_step(i):
            b = pool_d[i % npool]
            graphed(inputs_of(b), b[2])
    else:
        def dev_step(i):
            train_step(pool_d[i % npool], False)

    # ---- warm-up, then the device-resident timed region ---------------------------------------------------------
    for i in range(warmup):
        dev_step(i)
    sampler = ClockSampler(job.local_rank) if (sample_clocks and rank == 0) else None
    if sampler:
        sampler.start()
    n0 = _lib.launch_count()
    total_ms = job.timed(dev_step, steps)
    launches = (graphed.launches_per_step * steps) if graph_mode else (_lib.launch_count() - n0)
    clocks = sampler.stop() if sampler else None
    ms_per_step = total_ms / steps
    res = {"workload": workload, "desc": desc, "batch_per_gpu": B, "value": world * B / (ms_per_step * 1e-3),
           "ms_per_step": ms_per_step, "gpu_launches": int(launches), "clocks": clocks, "steps": steps,
           "launches_per_step": int(launches // max(steps, 1))}
    if dump and rank == 0:
        if graph_mode:
            outs, step_losses = graphed.outputs, graphed.losses
        else:
            outs, step_losses = last["outs"], last["losses"]
        res["dump"] = step_arrays(model, outs if isinstance(outs, tuple) else (outs,), step_losses)

    # ---- end-to-end: pinned host buffers, H2D inside the timed region, loss reads ------------------------------------
    if want_e2e:
        if graph_mode:
            # batch i+1 is copied from pinned host memory on a side stream while step i runs (DevicePrefetcher); every
            # step's inputs cross PCIe inside the timed region and both loss values are read back each step, the host
            # blocking on step i's values only after step i+1 has been enqueued (LossReader).
            reader = LossReader(2 if towers > 1 else 1, dev)
            e2e_state = {}

            def e2e_run(n):
                def host_batches():
                    for i in range(n):
                        hb = pool_h[i % npool]
                        yield (hb[0], hb[2]) if towers == 1 else hb
                pf = DevicePrefetcher(host_batches(), dev, reuse=e2e_state.get("pf"))
                e2e_state["pf"] = pf                         # the next "epoch" reuses its stream and device buffers
                for db in pf:
                    out = graphed(db[:-1], db[-1])
                    reader.push(out[1:])
                return reader.flush()

            e2e_run(2)
            job.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            e2e_run(steps)
            e1.record()
            job.barrier()
            e2e_ms = job.max_over_ranks(e0.elapsed_time(e1)) / steps
        else:
            def e2e_step(i):
                hb = pool_h[i % npool]
                db = tuple(t.to(dev, non_blocking=True) for t in hb)
                train_step(db, True)

            for i in range(2):
                e2e_step(i)
            e2e_ms = job.timed(e2e_step, steps) / steps
        h2d = sum(t.numel() * t.element_size() for t in pool_h[0][: (1 if towers == 1 else 2)]) + pool_h[0][2].numel() * 8
        # the PCIe leg on its own (pinned host -> device, nothing else running): when e2e ~= this, the step is link-bound
        probe_dst = [torch.empty_like(t, device=dev) for t in pool_h[0][: (1 if towers == 1 else 2)]]
        h2d_ms_alone = []
        for _ in range(3):
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for d, hsrc in zip(probe_dst, pool_h[0]):
                d.copy_(hsrc, non_blocking=True)
            e1.record()
            torch.cuda.synchronize()
            h2d_ms_alone.append(e0.elapsed_time(e1))
        del probe_dst
        res["e2e"] = {"value": world * B / (e2e_ms * 1e-3), "unit": "subjects/s", "ms_per_step": e2e_ms,
                      "h2d_bytes_per_step": int(h2d) * world, "d2h_bytes_per_step": (8 if towers > 1 else 4) * world,
                      "h2d_ms_alone": round(min(h2d_ms_alone), 4), "h2d_gbs_alone": round(h2d / min(h2d_ms_alone) / 1e6, 2),
                      "h2d_bytes_per_rank": int(h2d)}

    # ---- sustained: thousands of replays back to back, clocks recorded ---------------------------------------------
    if sustained_steps > 0 and graph_mode:
        s2 = ClockSampler(job.local_rank) if rank == 0 else None
        if s2:
            s2.start()
        ms = job.timed(dev_step, sustained_steps)
        c2 = s2.stop() if s2 else None
        res["sustained"] = {"steps": sustained_steps, "ms_per_step": ms / sustained_steps,
                            "value": world * B / (ms / sustained_steps * 1e-3), "unit": "subjects/s",
                            "seconds": round(ms * 1e-3, 2), "clocks": c2}

    # ---- roofline leg: CUDA events around every C-ABI launch (separate pass; not part of `value`) --------------------
    if want_roofline:
        peaks = measured_peaks()
        nprof = 3
        rec = {}
        for i in range(nprof):
            torch.cuda.synchronize()
            torch.cuda._sleep(int(1.5e8))                    # ~75 ms spin: the host enqueues the whole step behind it, so
            _lib.TIMER.start()                               # the events bracket back-to-back device execution
            train_step(pool_d[i % npool], False)
            r = _lib.TIMER.stop()
            if i == 0:
                continue                                     # first pass: warm-up of the timing path itself
            for t, (ms, n) in r.items():
                a = rec.get(t, (0.0, 0))
                rec[t] = (a[0] + ms, a[1] + n)
        nprof -= 1
        # dominant kernel family: the tcgen05 implicit-GEMM convolutions conv2.0 .. conv4.3 (fwd, dgrad, wgrad), the
        # layers SURVEY.md section 8d puts under the tensor roofline.  conv1.0 (Cin = 1, 26 FLOP/B) is HBM-bound and
        # is reported against the copy bandwidth below, together with the other block-1 passes.
        gemm_tags = ("tmf_conv3d_fwd", "tmf_conv3d_dgrad", "tmf_conv3d_wgrad")
        conv1_tags = ("tmf_conv1_fwd", "tmf_conv1_wgrad", "tmf_conv1_bwd_fused")
        gemm_ms = sum(v[0] for t, v in rec.items() if t.split("@")[0] in gemm_tags) / nprof
        conv1_ms = sum(v[0] for t, v in rec.items() if t.split("@")[0] in conv1_tags) / nprof
        flops = 0.0 if "dim" not in kwargs else conv_flops_per_subject(SHAPE, kwargs["dim"], towers, first_layer=False) * B
        flops_all = conv_flops_per_subject(SHAPE, kwargs["dim"], towers) * B
        achieved = flops / (gemm_ms * 1e-3) / 1e12
        achieved_all = flops_all / ((gemm_ms + conv1_ms) * 1e-3) / 1e12
        traffic = committed_traffic()
        hbm = {}
        for tag, nbytes in block1_bytes_per_subject(SHAPE, kwargs["dim"], towers).items():
            if tag in rec:
                ms = rec[tag][0] / nprof
                gbs = nbytes * B / (ms * 1e-3) / 1e9
                hbm[tag] = {"ms": round(ms, 4), "algorithmic_mb": round(nbytes * B / 1e6, 1), "achieved_gbs": round(gbs, 1),
                            "frac_of_hbm_peak": round(gbs / peaks["hbm_gbs"], 3)}
        res["roofline"] = {
            "bound": "tensor",
            "kernel": "conv3d implicit GEMM on tcgen05: fwd + dgrad + wgrad of conv2.0 .. conv4.3, both towers (18 launches per step)",
            "achieved": achieved, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s", "frac": achieved / peaks["bf16_tflops"],
            "peak_source": f"{peaks['source']} bf16 BURST (each launch is 20-230 us, event-timed on its own at full clock)",
            "frac_of_sustained_peak": achieved / peaks["bf16_tflops_sustained"],
            "traffic": traffic["dram_bytes_per_step"] if traffic else None,
            "traffic_source": traffic["source"] if traffic else None,
            "algorithmic_gflop_per_step": flops / 1e9, "conv_ms_per_step": gemm_ms,
            "timing": "CUDA events around each launch; launches enqueued behind a spin kernel (no host gaps inside the brackets)",
            "all_conv_incl_conv1": {"achieved": achieved_all, "frac": achieved_all / peaks["bf16_tflops"],
                                    "algorithmic_gflop_per_step": flops_all / 1e9, "ms_per_step": gemm_ms + conv1_ms,
                                    "note": "conv1.0 fwd and the fused block-1 backward (BN/LeakyReLU/MaxPool backward + conv1.0 "
                                            "wgrad) are HBM-bound passes; their whole time is counted here"},
            "hbm_bound_block1": {"peak_gbs": peaks["hbm_gbs"], "kernels": hbm}}
        res["breakdown"] = {t: round(rec[t][0] / nprof, 4) for t in sorted(rec)}   # ms per step per entry point (@L = layer)

    reducer.remove()
    del graphed, model, opt, reducer, pool_d, pool_h
    gc.collect()
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="both", choices=sorted(WORKLOADS) + ["both"],
                    help="both: model_ad is the headline, model_CNN_ad rides in `workloads`")
    ap.add_argument("--batch", type=int, default=8, help="subjects per GPU per step")
    ap.add_argument("--mode", default="graph", choices=["graph", "eager"],
                    help="graph: the step replayed as CUDA graphs (transmf_ad_b200.train.GraphedTrainStep); "
                         "eager: the reference's Python loop, one launch at a time")
    ap.add_argument("--optimizer", default="fused", choices=["fused", "torch"],
                    help="fused: transmf_ad_b200.optim.FusedAdam (one launch); torch: torch.optim.Adam as the reference builds it")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-roofline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the eager_dropin / sustained / c4 sub-records")
    ap.add_argument("--sustained-steps", type=int, default=2000)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the arrays the last timed step computed as DIR/<workload>.<name>.npy (at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl == "reference":
        ap.error("--dump-outputs records the CUDA path; --impl reference times the CPU port")
    if args.impl == "reference":
        run_reference_arm(args, int(os.environ.get("RANK", "0")))
        return
    args.warmup = max(args.warmup, 3)

    job = Job(args)
    rank, world = job.rank, job.world
    B = args.batch
    head_name = "ad" if args.workload == "both" else args.workload
    dump = args.dump_outputs is not None
    head = measure(job, head_name, B, args.steps, args.warmup, args.mode, args.optimizer, want_e2e=True,
                   want_roofline=(not args.no_roofline) and head_name != "mnet", sample_clocks=True,
                   sustained_steps=(args.sustained_steps if (world == 1 and not args.no_extras and args.mode == "graph") else 0),
                   dump=dump)
    dumped = {f"{head_name}.{k}": v for k, v in head.pop("dump", {}).items()}
    others = {}
    if args.workload == "both":
        r = measure(job, "cnn_ad", B, args.steps, args.warmup, args.mode, args.optimizer, want_e2e=True, want_roofline=False,
                    dump=dump)
        dumped.update({f"cnn_ad.{k}": v for k, v in r.pop("dump", {}).items()})
        others["cnn_ad"] = {k: r[k] for k in ("desc", "batch_per_gpu", "value", "ms_per_step", "e2e", "launches_per_step")}
    extras = {}
    if not args.no_extras and world == 1 and args.mode == "graph":
        r = measure(job, head_name, B, max(5, min(args.steps, 10)), 3, "eager", "torch", want_e2e=True, want_roofline=False)
        extras["eager_dropin"] = {"what": "the reference's unchanged loop on these modules: eager launches, torch.optim.Adam, "
                                          "host batches copied with .to(device), two .item() loss reads per step",
                                  "value": r["e2e"]["value"], "unit": "subjects/s", "ms_per_step": r["e2e"]["ms_per_step"],
                                  "device_resident_value": r["value"], "launches_per_step": r["launches_per_step"]}
    if not args.no_extras and world > 1 and args.mode == "graph" and 64 % world == 0:
        # BASELINE configs[3]: model_ad, global batch 64 data-parallel over the ranks (strong scaling; task pMCIsMCI only
        # changes labels).  Batch 64/N per GPU.
        r = measure(job, "ad", 64 // world, max(5, min(args.steps, 10)), 3, "graph", args.optimizer, want_e2e=True,
                    want_roofline=False)
        extras["c4"] = {"what": "BASELINE configs[3]: model_ad, global batch 64 split over the ranks (strong scaling)",
                        "global_batch": 64, "batch_per_gpu": 64 // world, "value": r["value"], "unit": "subjects/s",
                        "ms_per_step": r["ms_per_step"], "e2e": r["e2e"]}

    # ---- CPU baseline (rank 0, N = 1 only): BASELINE configs[0] ------------------------------------------------------
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        sps, mean_s, best = time_cpu_port("ad" if head_name == "ad" else head_name, CPU_SAMPLE_BATCH, 3, 1)
        cpu_baseline = {"value": sps, "unit": "subjects/s", "cores": torch.get_num_threads(), "kind": "port",
                        "best_step_value": best,
                        "sample": f"3 steps (after 1 warm-up) of batch {CPU_SAMPLE_BATCH} (BASELINE configs[0]) of the same workload, "
                                  "mean step, fwd+bwd+Adam, fp32 torch CPU; oracle/restatement.py (the reference is pure PyTorch, "
                                  "its kernels are ATen's)"}

    if rank == 0:
        if dump:
            print(f"[bench] --dump-outputs: {write_dump(args.dump_outputs, dumped)}", file=sys.stderr)
        graph_mode = args.mode == "graph"
        line = {
            "metric": METRIC, "value": head["value"], "unit": "subjects/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"{head['desc']}, batch {B}/GPU, volumes 91x109x91 fp32, Adam lr 1e-4",
                       "global_batch": B * world, "parallelism": f"dp{world}",
                       "conv_impl": os.environ.get("TMF_CONV_IMPL", "auto"),
                       "optimizer": "FusedAdam (tmf_adam_step)" if args.optimizer == "fused" else "torch.optim.Adam",
                       "mode": ("CUDA-graph replay of the whole step incl. the gradient all-reduce "
                                "(transmf_ad_b200.train.GraphedTrainStep); e2e adds DevicePrefetcher (H2D of batch i+1 on a side "
                                "stream) and LossReader (losses of step i read on the host after step i+1 is enqueued)")
                               if graph_mode else "eager launches",
                       "l2": "per-step working set (~0.2 GB/subject of activations) >> 126 MB L2; inputs rotate over a pool",
                       "library": library_hash(), "cpu_affinity": job.affinity},
            "e2e": head.get("e2e"), "gpu_launches": head["gpu_launches"], "clocks": head["clocks"],
            "roofline": head.get("roofline"), "cpu_baseline": cpu_baseline, "workloads": others or None,
            "sustained": head.get("sustained"), "eager_dropin": extras.get("eager_dropin"), "c4": extras.get("c4"),
            "breakdown": head.get("breakdown"),
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        job.dist.destroy_process_group()


if __name__ == "__main__":
    main()
