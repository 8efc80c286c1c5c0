"""AIR-ASR training driver: the reference trainer's loop (``train_air_pr.py:292-402``) on the captured data-parallel step.

    python -m mog_asr_b200.air.train -dn 13 -gm 100 -gne 10 -r results -k c2          (one GPU)
    torchrun --nproc_per_node 8 -m mog_asr_b200.air.train -dn 24 --global-batch 4096 -r results -k c4

Every step trains on a fresh batch of the on-device dataset (``DeviceMultiObjectDataset``): batch ``k`` of rank ``r`` is
``batch(k, B / world, r, world)``, so the stream is a function of the step index and a resumed run sees the batches the
uninterrupted one would have.  On a GPU the feed is part of the captured step: replay ``k`` pastes batch ``k + 1`` on a
side-stream branch while it trains on batch ``k`` (``Trainer.capture(feed=...)``).  The logged variables are summed on
the device inside the graph and read once per log interval (one JSON line per interval in ``<r>/<k>/log.jsonl``); every
``--test-every`` steps the test model and the detection metrics run on a fixed held-out set of 1000 canvases, sharded
over the ranks (``test.jsonl``); every ``--save-every`` steps rank 0 writes a checkpoint (``ckpt-<step>.pt``, the last
``--keep`` kept) with the model, Adam's state, the step index, the flags and config, and every rank's RNG states, from
which ``--resume`` continues.

``train`` takes the operators, the batch sources and the metrics as arguments, so the loop itself also runs on the CPU
with the oracle's operators (tests/test_train_driver.py)."""
from __future__ import annotations

import argparse
import dataclasses
import json
import os
import re
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

from .evaluate import evaluate_detection_sums, sums_to_means
from .model import config_from_flags
from .trainer import Trainer

REFERENCE_FLAGS = ("data", "dn", "ds", "gn", "gm", "gne", "gb", "gs", "ga", "zt")
TEST_SET_SIZE = 1000
TRAIN_SEED, TEST_SEED = 0, 1
LOG_FIELDS = ("loss", "elbo", "reconstruction", "pr_num", "num_min", "area", "out", "size", "overlap", "accuracy",
              "margin", "steps")
_SHARDED = 10   # the first ten fields are sums over the global batch divided by its size: summed over ranks when read


def parser() -> argparse.ArgumentParser:
    p = argparse.ArgumentParser(prog="python -m mog_asr_b200.air.train", allow_abbrev=False,
                                description="AIR-ASR training on the on-device dataset (train_air_pr.py:292-402)")
    p.add_argument("-data", default="mnist", help="mnist (50x50 canvases) or sprites (64x64)")
    p.add_argument("-dn", default="13", help="object counts, one digit each (one digit: a fixed count)")
    p.add_argument("-ds", default="", help="dataset name; containing 'bbox' selects box placement and the small size range")
    for f in ("gn", "gm", "gne", "gb", "gs", "ga"):
        p.add_argument("-" + f, type=float, default=0.0, help="ASR penalty weight (config_from_flags)")
    p.add_argument("-zt", type=float, default=0.1, help="z_pres Concrete temperature")
    p.add_argument("-r", default="results", help="results root")
    p.add_argument("-k", default="air", help="run name: the results folder is <r>/<k>")
    p.add_argument("-o", action="store_true", help="overwrite an existing results folder")
    p.add_argument("--global-batch", type=int, default=64, help="images per step over all ranks (BATCH_SIZE)")
    p.add_argument("--steps", type=int, default=100000, help="training steps in total (a resumed run counts the done ones)")
    p.add_argument("--sprites", default=None, help="[N, side, side] .npy of objects in [0, 1], e.g. MNIST digits")
    p.add_argument("--resume", action="store_true", help="continue from the newest checkpoint of the results folder")
    p.add_argument("--log-every", type=int, default=20)
    p.add_argument("--test-every", type=int, default=200)
    p.add_argument("--save-every", type=int, default=10000)
    p.add_argument("--keep", type=int, default=3, help="checkpoints kept (max_to_keep)")
    return p


def parse_args(argv=None):
    a = parser().parse_args(argv)
    for name in ("global_batch", "steps", "log_every", "test_every", "save_every", "keep"):
        if getattr(a, name) <= 0:
            raise SystemExit(f"--{name.replace('_', '-')} must be positive")
    return a


def make_config(args, captured: bool):
    """``config_from_flags`` of the reference flags; the captured step runs ``max_steps`` iterations with the reference's
    trip count counted on the device (``AIRConfig.reference_trip_count``), the eager one the reference loop itself"""
    flags = {f: getattr(args, f) for f in REFERENCE_FLAGS}
    return config_from_flags(always_max_steps=captured, reference_trip_count=captured, **flags)


def dataset_mode(args) -> str:
    return "bbox" if "bbox" in args.ds else "pixel"


def device_datasets(args, cfg, device):
    """(training set, held-out set): the feeder with the config's canvas, counts and size range, seeded apart"""
    from ..dataset import DeviceMultiObjectDataset, default_sprites
    sprites = default_sprites() if args.sprites is None else np.load(args.sprites)
    lo, hi = (int(v) for v in cfg.constrains_area_minmax)
    mk = lambda seed: DeviceMultiObjectDataset(sprites, cfg.canvas_size, tuple(cfg.constrains_num), (lo, hi),
                                               mode=dataset_mode(args), seed=seed, device=device)
    return mk(TRAIN_SEED), mk(TEST_SEED)


def make_feed(ds, B, rank, world):
    """``feed(k)``: the clamped images and the counts of ``ds.batch(k, B, rank, world)``; ``k`` an int or a 0-d int64 device
    tensor (then the placement reads the index when it runs, and a captured graph can advance it)"""
    def feed(k):
        placed = ds.place((k * world + rank) * B, B)
        return dict(images=torch.clamp(ds.paste(*placed), 0.0, 1.0), num=placed[0])
    return feed


class LogAccumulator:
    """Per-step log variables added into one float64 device vector (capturable); read and reset once per interval."""

    def __init__(self, device, global_batch, process_group=None):
        self.buf = torch.zeros(len(LOG_FIELDS), dtype=torch.float64, device=device)
        self.n, self.pg = global_batch, process_group
        self.count = 0

    def add(self, out, batch):
        f64 = lambda t: t.detach().to(torch.float64)
        margin = f64(out["margin"]).reshape(1)
        steps = out["steps"]
        steps = (f64(steps) if isinstance(steps, torch.Tensor) else torch.full((), float(steps), dtype=torch.float64,
                                                                                 device=self.buf.device)).reshape(1)
        digits = out["rec_num_digits"]
        correct = (digits == batch["num"].to(digits.device, digits.dtype)).to(torch.float64).sum().reshape(1)
        row = torch.cat([f64(out["loss"]).reshape(1) - margin,          # the rank's share: sum_b(...) / n (model.py)
                         f64(out["elbo"]).sum().reshape(1) / self.n, f64(out["recon"]).sum().reshape(1) / self.n,
                         f64(out["components"]).sum(0) / self.n, correct / self.n, margin, steps])
        self.buf.add_(row)

    def read(self):
        """means over the steps added since the last read (every rank gets them; one all-reduce)"""
        v = self.buf.clone()
        if self.pg is not None:
            dist.all_reduce(v[:_SHARDED], group=self.pg)   # (a view: all_reduce writes into it)
        v = v.cpu()
        v[0] += v[LOG_FIELDS.index("margin")]
        means = (v / max(self.count, 1)).tolist()
        self.buf.zero_()
        self.count = 0
        return dict(zip(LOG_FIELDS, means))


def _rng_state(trainer):
    st = dict(trainer_generator=trainer.gen.get_state())
    if trainer.device.type == "cuda":
        g = torch.cuda.default_generators[trainer.device.index or 0]
        st.update(cuda_seed=int(g.initial_seed()), cuda_offset=int(g.get_offset()), cuda_state=g.get_state())
    else:
        st.update(cpu_state=torch.get_rng_state())
    return st


def _set_rng_state(trainer, st):
    trainer.gen.set_state(st["trainer_generator"].cpu())      # (generator states are host byte tensors)
    if trainer.device.type == "cuda":
        g = torch.cuda.default_generators[trainer.device.index or 0]
        g.set_state(st["cuda_state"].cpu())
        if int(g.get_offset()) != st["cuda_offset"] or int(g.initial_seed()) != st["cuda_seed"]:
            raise RuntimeError("restoring the CUDA generator's seed and offset failed")
    else:
        torch.set_rng_state(st["cpu_state"].cpu())


def _plain(x):
    if isinstance(x, dict):
        return {k: _plain(v) for k, v in x.items()}
    if isinstance(x, (list, tuple)):
        return [_plain(v) for v in x]
    return x


def checkpoint_path(folder, step):
    return os.path.join(folder, f"ckpt-{step:08d}.pt")


def checkpoints(folder):
    names = sorted(f for f in os.listdir(folder) if re.fullmatch(r"ckpt-\d{8}\.pt", f)) if os.path.isdir(folder) else []
    return [os.path.join(folder, f) for f in names]


def save_checkpoint(folder, step, trainer, args, cfg, acc, keep, process_group=None):
    """every rank contributes its RNG states and its log sums (per-rank shares until the interval's read); rank 0 writes
    (to a temporary name, then renamed) and prunes to ``keep``"""
    mine = dict(rng=_rng_state(trainer), log_buffer=acc.buf.cpu())
    if process_group is not None:
        ranks = [None] * dist.get_world_size(process_group)
        dist.all_gather_object(ranks, mine, group=process_group)
    else:
        ranks = [mine]
    if trainer.rank != 0:
        return
    with torch.no_grad():
        ck = dict(step=int(step), model=trainer.model.state_dict(), adam_m=[m.clone() for m in trainer.m],
                  adam_v=[v.clone() for v in trainer.v], t=int(trainer.t), t_dev=trainer.t_dev.clone(),
                  flags=_plain(vars(args)), config=_plain(dataclasses.asdict(cfg)), rng=[r["rng"] for r in ranks],
                  log_buffer=[r["log_buffer"] for r in ranks], log_count=int(acc.count))
    path = checkpoint_path(folder, step)
    torch.save(ck, path + ".tmp")
    os.replace(path + ".tmp", path)
    for old in checkpoints(folder)[:-keep]:
        os.remove(old)


def load_checkpoint(path, trainer, acc):
    """parameters, Adam state and step count, and this rank's own log sums; returns the checkpoint (RNG states are restored
    by the caller, after capture)"""
    ck = torch.load(path, map_location=trainer.device, weights_only=True)
    if len(ck["rng"]) != trainer.world:
        raise RuntimeError(f"{path} holds {len(ck['rng'])} ranks' states; this run has {trainer.world} ranks")
    with torch.no_grad():
        trainer.model.load_state_dict(ck["model"])
        for dst, src in zip(trainer.m + trainer.v, ck["adam_m"] + ck["adam_v"]):
            dst.copy_(src)
        trainer.t_dev.copy_(ck["t_dev"])
        acc.buf.copy_(ck["log_buffer"][trainer.rank])
    trainer.t, acc.count = ck["t"], ck["log_count"]
    return ck


def held_out_pass(trainer, test_source, metrics=None, test_noise=None, size=TEST_SET_SIZE):
    """canvases ``0 .. size - 1`` of the held-out set, sharded evenly over the ranks and scored; returns the means over the
    whole set (one all-reduce of the per-image sums)"""
    world, rank = trainer.world, trainer.rank
    if size % world:
        raise ValueError(f"the test set of {size} canvases does not split evenly over {world} ranks")
    n = size // world
    batch = test_source(0, n, rank, world)          # canvases rank*n .. rank*n + n - 1
    noise = None if test_noise is None else test_noise(rank * n, rank * n + n)
    sums = evaluate_detection_sums(trainer.model, batch, noise=noise,
                                   any_reduce=trainer._any_reduce if trainer.pg is not None else None, metrics=metrics)
    if trainer.pg is not None:
        dist.all_reduce(sums, group=trainer.pg)
    return sums_to_means(sums.cpu())


def _results_folder(args, rank, process_group, test_size):
    """checks the run's set-up on rank 0 and makes every rank stop on the same error before any collective waits for it"""
    folder = os.path.join(args.r, args.k)
    world = dist.get_world_size(process_group) if process_group is not None else 1
    error = None
    if rank == 0:
        if args.global_batch % world:
            error = f"--global-batch {args.global_batch} does not split over {world} ranks"
        elif test_size % world:
            error = f"the test set of {test_size} canvases does not split evenly over {world} ranks"
        elif os.path.exists(folder) and os.listdir(folder) and not (args.o or args.resume):
            error = f"{folder} exists: pass -o to overwrite it or --resume to continue it"
        elif args.resume and not checkpoints(folder):
            error = f"--resume: no checkpoint in {folder}"
    if process_group is not None:
        box = [error]
        dist.broadcast_object_list(box, src=0, group=process_group)
        error = box[0]
    if error is not None:
        raise SystemExit(error)
    if rank == 0:
        os.makedirs(folder, exist_ok=True)
        if args.o and not args.resume:
            for f in checkpoints(folder) + [os.path.join(folder, n) for n in ("log.jsonl", "test.jsonl")]:
                if os.path.exists(f):
                    os.remove(f)
    if process_group is not None:
        dist.barrier(process_group)
    return folder


def train(args, device, process_group=None, ops=None, source=None, test_source=None, metrics=None, test_noise=None,
          dtype=torch.float32, out=sys.stdout, test_size=TEST_SET_SIZE, feed_in_graph=True):
    """The loop.  Default: the product operators, the captured step with the feed inside it, the device dataset and the
    device detection metrics.  ``ops`` given: the eager step with those operators (the reference loop condition), fed
    by ``source(index, batch_size, rank, world)`` (a dict with ``images`` and ``num``); ``test_source`` likewise for the
    held-out set, ``metrics`` in place of ``detection.detection_metrics``, ``test_noise(lo, hi)`` the test model's draws
    for canvases ``lo .. hi - 1``.  ``test_size``: canvases of the held-out set.  ``feed_in_graph=False`` feeds the captured
    step eagerly before each replay (the baseline ``tools/train_driver_bench.py`` times the in-graph feed against).
    Returns the trainer."""
    device = torch.device(device)
    world = dist.get_world_size(process_group) if process_group is not None else 1
    rank = dist.get_rank(process_group) if process_group is not None else 0
    captured = ops is None
    if captured and device.type != "cuda":
        raise RuntimeError("the product step needs a CUDA device: there is no CPU fallback (pass ops= for the oracle)")
    folder = _results_folder(args, rank, process_group, test_size)
    B = args.global_batch // world
    cfg = make_config(args, captured)
    if rank == 0:
        header = dict(args=_plain(vars(args)), config=_plain(dataclasses.asdict(cfg)), world=world)
        print(json.dumps(header), file=out, flush=True)
        with open(os.path.join(folder, "config.json"), "w") as f:
            json.dump(header, f, indent=1)
    tr = Trainer(cfg, device, process_group=process_group, global_batch=args.global_batch, ops=ops, dtype=dtype)
    acc = LogAccumulator(device, args.global_batch, process_group)

    if captured:
        train_ds, test_ds = device_datasets(args, cfg, device)
        test_source = test_ds.batch
        tr.capture(B, feed=make_feed(train_ds, B, rank, world), on_step=acc.add, feed_in_graph=feed_in_graph)

        def step(k):
            tr.step_graph()
            acc.count += 1
    else:
        def step(k):
            b = source(k, B, rank, world)
            o = tr.step(torch.clamp(b["images"], 0.0, 1.0).to(device, dtype))
            acc.add(o, b)
            acc.count += 1

    start = 0
    found = checkpoints(folder) if args.resume else []
    if found:
        ck = load_checkpoint(found[-1], tr, acc)
        start = ck["step"]
        _set_rng_state(tr, ck["rng"][rank])     # after capture: capturing reseeds the default CUDA generator
    if captured:
        tr.start_feed(start)
    gpu = torch.cuda.get_device_name(device) if device.type == "cuda" else "cpu"
    t0, k0 = time.perf_counter(), start
    for k in range(start, args.steps):
        step(k)
        done = k + 1
        if done % args.log_every == 0:
            means = acc.read()
            dt = time.perf_counter() - t0
            line = dict(step=done, **means, images_per_sec=args.global_batch * (done - k0) / dt, gpu=gpu)
            if rank == 0:
                with open(os.path.join(folder, "log.jsonl"), "a") as f:
                    f.write(json.dumps(line) + "\n")
                print(json.dumps(line), file=out, flush=True)
            t0, k0 = time.perf_counter(), done
        if done % args.test_every == 0:
            res = held_out_pass(tr, test_source, metrics, test_noise, test_size)
            line = dict(step=done, **{k_: (v.tolist() if v.dim() else float(v)) for k_, v in res.items()})
            if rank == 0:
                with open(os.path.join(folder, "test.jsonl"), "a") as f:
                    f.write(json.dumps(line) + "\n")
            t0, k0 = time.perf_counter(), done
        if done % args.save_every == 0 or done == args.steps:
            save_checkpoint(folder, done, tr, args, cfg, acc, args.keep, process_group)
            t0, k0 = time.perf_counter(), done
    if device.type == "cuda":
        torch.cuda.synchronize(device)
    return tr


def main(argv=None):
    args = parse_args(argv)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("mog_asr_b200.air.train needs a CUDA device: there is no CPU fallback")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    pg = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        pg = dist.group.WORLD
    try:
        train(args, dev, process_group=pg)
    finally:
        if pg is not None:
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
