"""AIR-ASR training-step throughput (BASELINE configs 2-4) on synthetic canvases: images/sec."""
from __future__ import annotations

import os
import time

import numpy as np
import torch
import torch.distributed as dist

from .. import synth
from .model import config_from_flags
from .trainer import Trainer

CONFIGS = {
    # name: (flags, global batch)
    "C2": (dict(data="mnist", dn="13", gm=100.0, gne=10.0), 64),
    "C3": (dict(data="sprites", dn="3", ds="bbox20k", gb=1.0, gs=10.0, ga=20.0), 256),
    "C4": (dict(data="mnist", dn="24"), 4096),
}


_DATASETS = {}


def synthetic_batch(cfg, batch, seed, device):
    """``[batch, canvas*canvas]`` canvases in [0, 1].  On a GPU they come from the on-device feeder
    (``mog_asr_b200/dataset.py``: placement kernel + the sampler's own write direction); the numpy generator of
    ``synth.py`` serves the CPU tests."""
    dev = torch.device(device)
    if dev.type == "cuda":
        from ..dataset import DeviceMultiObjectDataset, default_sprites
        key = (str(dev), cfg.canvas_size, tuple(cfg.constrains_num), tuple(cfg.constrains_area_minmax))
        if key not in _DATASETS:
            lo, hi = (int(v) for v in cfg.constrains_area_minmax)
            _DATASETS[key] = DeviceMultiObjectDataset(default_sprites(256, 28, seed=0), cfg.canvas_size, tuple(cfg.constrains_num),
                                                      (lo, hi), mode="disjoint", seed=1234, device=dev)
        return torch.clamp(_DATASETS[key].batch(seed, batch)["images"], 0.0, 1.0)
    canv, _ = synth.multi_object_canvases(batch, cfg.canvas_size, 28, tuple(cfg.constrains_num), seed=seed)
    return torch.tensor(np.clip(canv, 0.0, 1.0).reshape(batch, -1), device=device)


def run(name, device, steps=20, warmup=5, process_group=None, always_max_steps=False, graph=False, per_rank_batch=None,
        reference_trip_count=False):
    """Returns dict(images_per_sec, ms_per_step, global_batch, per_rank_batch, mean loop steps).  ``per_rank_batch``
    overrides the config's fixed global batch with ``per_rank_batch * world`` (weak scaling).  ``reference_trip_count``
    (with ``always_max_steps``): the regularisers and the step count of the reference loop, counted on the device; the
    mean loop steps are then the reference's trip counts, summed on the device and read once after the timed loop."""
    flags, gbatch = CONFIGS[name]
    world = dist.get_world_size(process_group) if process_group is not None else 1
    rank = dist.get_rank(process_group) if process_group is not None else 0
    if per_rank_batch is not None:
        gbatch = per_rank_batch * world
    cfg = config_from_flags(always_max_steps=always_max_steps, reference_trip_count=reference_trip_count, **flags)
    local = gbatch // world
    tr = Trainer(cfg, device, process_group=process_group, global_batch=gbatch)
    # a few distinct resident batches, cycled (the reference feeds from a shuffle queue)
    batches = [synthetic_batch(cfg, local, 100 * rank + k, device) for k in range(4)]
    step_fn = tr.step
    if graph:
        tr.capture(local)
        step_fn = tr.step_graph
    for k in range(warmup):
        step_fn(batches[k % 4])
    torch.cuda.synchronize(device)
    if process_group is not None:
        dist.barrier(process_group)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    T = 0
    e0.record()
    for k in range(steps):
        T = T + step_fn(batches[k % 4])["steps"]      # a device tensor with reference_trip_count: no host read per step
    e1.record()
    torch.cuda.synchronize(device)
    T = int(T)
    ms = e0.elapsed_time(e1) / steps
    if process_group is not None:
        t = torch.tensor([ms], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=process_group)
        ms = float(t.item())
    kernels_per_step = None
    try:   # one profiled step: how many kernels the step is (the chain's length bounds strong scaling, DESIGN.md section 7)
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            step_fn(batches[0])
            torch.cuda.synchronize(device)
        kernels_per_step = sum(1 for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
                               and not e.name.lower().startswith(("memcpy", "memset")))
    except Exception:
        pass
    if reference_trip_count:
        mode = ("CUDA graph" if graph else "eager") + ", max_steps iterations, reference trip count (device-counted)"
    elif always_max_steps:
        mode = "CUDA graph, fixed max_steps" if graph else "eager, fixed max_steps"
    else:
        mode = "eager, reference loop condition (host-checked any)"
    return dict(config=name, images_per_sec=gbatch / (ms * 1e-3), ms_per_step=ms, global_batch=gbatch, kernels_per_step=kernels_per_step,
                graph_branches=(os.environ.get("MOG_AIR_STREAMS", "1") != "0") if graph else False,
                per_rank_batch=local, n_gpus=world, mean_loop_steps=T / steps, grad_floats=tr.num_gradient_floats(),
                mode=mode)


class GlobalSeededNoise:
    """``noise(kind, step, shape)`` for data-parallel checks: the draw for the GLOBAL batch comes from a CPU generator seeded by
    (seed, kind, step) and the rank's rows are cut out, so that any sharding of the batch sees the same numbers."""
    _KIND = {"shift": 1, "scale": 2, "vae": 3, "concrete": 4}

    def __init__(self, seed, global_batch, lo, hi, device):
        self.seed, self.B, self.lo, self.hi, self.device = seed, global_batch, lo, hi, device

    def __call__(self, kind, step, shape):
        g = torch.Generator().manual_seed(self.seed * 1000 + self._KIND[kind] * 100 + step)
        full = (self.B,) + tuple(shape[1:])
        t = torch.rand(full, generator=g).clamp_(1e-4, 1 - 1e-4) if kind == "concrete" else torch.randn(full, generator=g)
        return t[self.lo:self.hi].to(self.device)


def dp_check(device, process_group, global_batch=64, seed=31, ops_factory=None):
    """Multi-GPU correctness of the training step on the hardware it runs on (SURVEY section 4: "1/2/4/8-GPU gradient equality
    vs 1-GPU at the same global batch"): config C2 (``-dn 13 -gm 100 -gne 10``: the ``[T]`` column-sum all-reduce of the marginal
    count penalty runs, air_number_bbox_location.py:982), ``global_batch`` images sharded over the ranks, identical noise per
    image on any sharding.  The all-reduced flat gradient is compared with the single-process gradient of the whole batch
    (computed on every rank), per parameter tensor, relative to that tensor's largest entry.  (``ops_factory(process_group,
    global_batch)`` replaces the product operators -- the CPU test of this function runs it over gloo.)

    Two reconstruction terms: the verdict (``max_rel_diff``, ``ok``) uses a squared-error term through the same graph, because the
    reference's cross-entropy (:954-959) has gradients of 1e10 wherever the canvas is 0 under an object pixel: the library GEMMs
    pick different tiles for a shard than for the whole batch, their sums differ in the last bit, and that term amplifies the
    difference to O(0.1) of a gradient entry in ANY fp32 implementation (tests/test_air_model.py has the same split).  The
    cross-entropy figures are reported beside it (``with_reference_cross_entropy``), not judged.

    A second pass runs the reference's loop form (``while any(stop_sum < thr)``, :386-390) and checks that every rank executed
    the same number of iterations as the single process (the one-flag ``any`` all-reduce)."""
    world, rank = dist.get_world_size(process_group), dist.get_rank(process_group)
    flags = CONFIGS["C2"][0]
    lo, hi = rank * global_batch // world, (rank + 1) * global_batch // world
    out = dict(config="C2 flags, global batch %d over %d ranks" % (global_batch, world))
    mse = lambda x, r: ((x - r) ** 2).sum(1) * 50.0
    mk = (lambda pg: None) if ops_factory is None else (lambda pg: ops_factory(pg, global_batch))

    def compare(amx, recon_fn):
        cfg = config_from_flags(always_max_steps=amx, **flags)
        images = synthetic_batch(cfg, global_batch, 4242, device)            # same canvases on every rank (seeded feeder)
        dp = Trainer(cfg, device, process_group=process_group, global_batch=global_batch, seed=seed, ops=mk(process_group))
        o_dp = dp.forward_backward(images[lo:hi], noise=GlobalSeededNoise(7, global_batch, lo, hi, device), recon_loss_fn=recon_fn)
        dp.reduce_gradients()
        one = Trainer(cfg, device, process_group=None, global_batch=global_batch, seed=seed, ops=mk(None))
        o_one = one.forward_backward(images, noise=GlobalSeededNoise(7, global_batch, 0, global_batch, device), recon_loss_fn=recon_fn)
        worst, worst_name, off = 0.0, "", 0
        for name, p in one.model.named_parameters():
            n = p.numel()
            a, b = one.flat_grad[off:off + n], dp.flat_grad[off:off + n]
            off += n
            scale = float(a.abs().max())
            if scale > 0:
                d = float((a - b).abs().max()) / scale
                if d > worst:
                    worst, worst_name = d, name
        local = (o_dp["loss"].detach() - o_dp["margin"]).reshape(1).clone()
        dist.all_reduce(local, group=process_group)
        loss_dp = float(local) + float(o_dp["margin"])
        steps = torch.tensor([o_dp["steps"]], device=device)
        gathered = [torch.zeros_like(steps) for _ in range(world)]
        dist.all_gather(gathered, steps, group=process_group)
        trip = [int(t) for t in gathered]
        w = torch.tensor([worst], device=device, dtype=torch.float64)
        dist.all_reduce(w, op=dist.ReduceOp.MAX, group=process_group)
        return dict(max_rel_diff=float(w), worst_parameter=worst_name, loss_dp=loss_dp, loss_single=float(o_one["loss"].detach()),
                    loss_rel_diff=abs(loss_dp - float(o_one["loss"].detach())) / max(abs(float(o_one["loss"].detach())), 1e-30),
                    trip_counts=trip, trip_count_single=int(o_one["steps"]),
                    same_trip_count=len(set(trip)) == 1 and trip[0] == int(o_one["steps"]))

    for mode, amx in (("fixed_trip_count", True), ("reference_loop", False)):
        out[mode] = compare(amx, mse)
    out["with_reference_cross_entropy"] = compare(True, None)
    out["max_rel_diff"] = max(out[m]["max_rel_diff"] for m in ("fixed_trip_count", "reference_loop"))
    out["ok"] = bool(out["max_rel_diff"] <= 2e-3 and all(out[m]["same_trip_count"] for m in ("fixed_trip_count", "reference_loop")))
    return out
