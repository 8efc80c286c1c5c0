"""One AIR-ASR training step, optionally data-parallel.

Reference: ``AIRModel.training`` = Adam(lr).apply_gradients after per-variable ``inf -> 0``, ``nan -> 0``,
``clip_by_norm(g, gradient_clipping_norm)`` (``air/air_number_bbox_location.py:1094-1122``); the host loop
``train_air_pr.py:292-295`` runs one such step per ``sess.run``.

Data parallelism (absent from the reference, SURVEY 2.3): the batch is sharded across ranks, parameters and
Adam state are replicated, and the step has exactly one exchange: an NCCL all-reduce(sum) of the flat fp32
gradient buffer *before* the per-variable post-processing (``:1100-1111``), plus the ``[T]`` column sums of
the marginal count penalty (``:982``) and a one-flag ``any`` per loop iteration (``:389``).  With
``AIRConfig.reference_trip_count`` the column sums travel with the per-step active counts (``[2T]`` floats) and there is
no per-iteration exchange: the trip count is derived on the device.
"""
from __future__ import annotations

from typing import Optional

import torch
import torch.distributed as dist

from .model import AIRConfig, AIRModel, CudaOps


class Trainer:
    def __init__(self, cfg: AIRConfig, device, process_group=None, global_batch: Optional[int] = None, seed: int = 1235,
                 ops=None, dtype=torch.float32, defer_weight_grads=True):
        self.cfg, self.device, self.pg = cfg, torch.device(device), process_group
        self.world = dist.get_world_size(process_group) if process_group is not None else 1
        self.rank = dist.get_rank(process_group) if process_group is not None else 0
        self.seed = seed
        self.global_batch = global_batch
        torch.manual_seed(seed)                       # identical initial parameters on every rank
        if ops is None:
            ops = CudaOps(process_group=process_group, global_batch=global_batch)
        self.model = AIRModel(cfg, ops).to(self.device, dtype)   # fp32 is the product; fp64 only for test oracles
        self.defer_weight_grads = defer_weight_grads
        self.params = [p for p in self.model.parameters()]
        # flat gradient bucket: every p.grad is a view into it -> one all-reduce per step
        n = sum(p.numel() for p in self.params)
        self.flat_grad = torch.zeros(n, dtype=dtype, device=self.device)
        off = 0
        for p in self.params:
            p.grad = self.flat_grad[off:off + p.numel()].view_as(p)
            off += p.numel()
        self.grads = [p.grad for p in self.params]
        self.m = [torch.zeros_like(p) for p in self.params]
        self.v = [torch.zeros_like(p) for p in self.params]
        self.t = 0
        self.t_dev = torch.zeros((), dtype=torch.float64, device=self.device)
        self.graph = None
        self._noise_bank = {}
        self.beta1, self.beta2, self.eps = 0.9, 0.999, 1e-8   # tf.train.AdamOptimizer defaults
        self.gen = torch.Generator(device=self.device)
        self.gen.manual_seed(seed + 1 + (dist.get_rank(process_group) if process_group is not None else 0))

    def num_gradient_floats(self) -> int:
        return self.flat_grad.numel()

    def _noise(self, kind, step, shape, generator="own"):
        """All loop iterations' draws of one kind come from a single RNG launch per training step."""
        bank = self._noise_bank
        if kind not in bank:
            full = (self.cfg.max_steps,) + tuple(shape)
            gen = self.gen if generator == "own" else None
            bank[kind] = (torch.rand(full, device=self.device, generator=gen) if kind == "concrete"
                          else torch.randn(full, device=self.device, generator=gen))
        return bank[kind][step]

    def _any_reduce(self, flag):
        if self.pg is None:
            return flag
        f = flag.to(torch.int32)
        dist.all_reduce(f, op=dist.ReduceOp.MAX, group=self.pg)
        return f

    def forward_backward(self, images, noise=None, recon_loss_fn=None):
        B = images.shape[0]
        nglobal = self.global_batch if self.global_batch is not None else B * self.world
        self.flat_grad.zero_()
        self._noise_bank = {}
        self.model.set_deferred_weight_grads(self.defer_weight_grads)
        out = self.model(images, noise=noise or self._noise, any_reduce=self._any_reduce if self.pg is not None else None,
                         global_batch=nglobal, recon_loss_fn=recon_loss_fn)
        out["loss"].backward()
        if self.defer_weight_grads:
            self.model.flush_weight_grads()   # one GEMM per layer over all loop iterations' rows
        return out

    def reduce_gradients(self):
        if self.pg is not None and self.world > 1:
            dist.all_reduce(self.flat_grad, op=dist.ReduceOp.SUM, group=self.pg)

    def clean_and_clip(self):
        """:1100-1111: per variable ``inf -> 0``, ``nan -> 0``, then ``tf.clip_by_norm(g, gradient_clipping_norm)``
        (``g * clip / max(||g||, clip)``); only when a clipping norm is configured, like the reference."""
        c = self.cfg.gradient_clipping_norm
        if c is None:
            return
        torch.nan_to_num_(self.flat_grad, nan=0.0, posinf=0.0, neginf=0.0)
        norms = torch.stack(torch._foreach_norm(self.grads))           # all 50 scales in three small kernels
        scales = c / torch.clamp(norms, min=c)
        torch._foreach_mul_(self.grads, list(scales.unbind(0)))

    def postprocess_and_apply(self):
        """:1100-1111 per-variable inf/nan -> 0 and clip_by_norm, then TF's Adam update
        ``lr_t = lr*sqrt(1-b2^t)/(1-b1^t); var -= lr_t * m / (sqrt(v) + eps)``.  The step counter lives on the
        device so the whole update is CUDA-graph capturable."""
        self.clean_and_clip()
        self.t += 1
        b1, b2 = self.beta1, self.beta2
        self.t_dev += 1.0
        lr_t = self.cfg.learning_rate * torch.sqrt(1.0 - torch.pow(b2, self.t_dev)) / (1.0 - torch.pow(b1, self.t_dev))
        torch._foreach_mul_(self.m, b1); torch._foreach_add_(self.m, self.grads, alpha=1.0 - b1)
        torch._foreach_mul_(self.v, b2); torch._foreach_addcmul_(self.v, self.grads, self.grads, value=1.0 - b2)
        denom = torch._foreach_sqrt(self.v)
        torch._foreach_add_(denom, self.eps)
        upd = torch._foreach_div(self.m, denom)
        torch._foreach_mul_(upd, -lr_t.to(self.flat_grad.dtype))
        with torch.no_grad():
            torch._foreach_add_(self.params, upd)

    # ---- CUDA-graph mode: the ~1500 small launches of one step replayed as one graph ------------------------
    def capture(self, batch_size: int, feed=None, on_step=None, feed_in_graph=True):
        """Capture forward + backward + all-reduce + update for a fixed local batch size.  Needs
        ``cfg.always_max_steps`` (the reference's data-dependent trip count, :386-390, needs a host decision per
        iteration and cannot be captured; ``cfg.reference_trip_count`` restores its objective inside the graph).  Noise comes from the default CUDA generator (graph-safe).

        ``feed(index)`` (optional) makes the trainer fetch its own batches: it returns a dict with ``images`` ``[B, cs*cs]``
        and any labels (tensors of fixed shape) for the step index ``index``, an int or a 0-d int64 device tensor read at
        run time.  ``step_graph()`` then takes no images: it trains on batch ``feed_step`` and advances the index.  With
        ``feed_in_graph`` the graph itself pastes batch ``k + 1`` on a side-stream branch while the step trains on batch
        ``k`` (double-buffered: the branch rejoins before the next batch is copied in); otherwise every ``step_graph``
        feeds eagerly on the current stream before the replay.  ``on_step(out, batch)`` (optional) is captured after the
        step, on the step's outputs and the batch it trained on (``static_batch``)."""
        if not self.cfg.always_max_steps:
            raise ValueError("graph capture needs AIRConfig.always_max_steps=True")
        cs2 = self.cfg.canvas_size ** 2
        self._feed, self._feed_in_graph = feed, bool(feed_in_graph)
        if feed is None:
            self.static_images = torch.zeros((batch_size, cs2), device=self.device)
            self.static_batch = dict(images=self.static_images)
        else:
            self.static_batch = {k: v.clone() for k, v in feed(0).items()}
            self.static_images = self.static_batch["images"]
            if tuple(self.static_images.shape) != (batch_size, cs2):
                raise ValueError(f"feed(k)['images'] must be [{batch_size}, {cs2}]")
            self.feed_k = 0
            self.feed_step = torch.zeros((), dtype=torch.int64, device=self.device)
        noise = lambda kind, step, shape: self._noise(kind, step, shape, generator="default")   # graph-safe default generator
        # The warm-up runs real steps (allocator, cuBLAS handles, NCCL): snapshot the training state first and put it
        # back afterwards, so that capturing changes neither the parameters nor Adam's moments / step count.
        with torch.no_grad():
            snap = [[t.clone() for t in ts] for ts in (self.params, self.m, self.v)]
        t_host, t_dev = self.t, self.t_dev.clone()
        # the captured graph draws from the default CUDA generator: give every rank its own stream of draws, like
        # the eager path's per-rank generator (identical seeds would repeat the same noise on every batch shard)
        torch.cuda.manual_seed(self.seed + 1 + self.rank)
        side = torch.cuda.Stream(self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(side):
            for _ in range(3):
                self.step(self.static_images, noise=noise)
                if feed is not None:
                    feed(self.feed_step)      # (reads index 0; loads the feed's kernels before capture)
        torch.cuda.current_stream(self.device).wait_stream(side)
        torch.cuda.synchronize(self.device)
        with torch.no_grad():
            for ts, saved in zip((self.params, self.m, self.v), snap):
                for t, s0 in zip(ts, saved):
                    t.copy_(s0)
            self.t_dev.copy_(t_dev)
        self.t = t_host
        self.flat_grad.zero_()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            nxt = None
            if feed is not None and self._feed_in_graph:
                main = torch.cuda.current_stream(self.device)
                self._feed_stream = self.__dict__.get("_feed_stream") or torch.cuda.Stream(self.device)
                self._feed_stream.wait_stream(main)
                with torch.cuda.stream(self._feed_stream):
                    nxt = feed(self.feed_step + 1)
            self.static_out = self.step(self.static_images, noise=noise)
            if on_step is not None:
                on_step(self.static_out, self.static_batch)
            if nxt is not None:
                main.wait_stream(self._feed_stream)
                for k, v in self.static_batch.items():
                    v.copy_(nxt[k])
                self.feed_step += 1
                self._feed_keep = nxt   # allocated on the branch: kept for the graph's lifetime
        self.t = t_host          # (tracing the step bumped the host-side counter; nothing ran)
        return self

    def start_feed(self, k: int):
        """With a ``feed``: the next ``step_graph`` trains on batch ``k``"""
        self.feed_k = int(k)
        self.feed_step.fill_(self.feed_k)
        if self._feed_in_graph:
            for key, v in self._feed(self.feed_k).items():
                self.static_batch[key].copy_(v)

    def step_graph(self, images=None):
        if self._feed is None:
            self.static_images.copy_(images, non_blocking=True)
        elif not self._feed_in_graph:
            for key, v in self._feed(self.feed_k).items():
                self.static_batch[key].copy_(v)
        self.graph.replay()
        if self._feed is not None:
            self.feed_k += 1
            if not self._feed_in_graph:
                self.feed_step += 1
        self.t += 1
        return self.static_out

    def step(self, images, noise=None):
        out = self.forward_backward(images, noise)
        self.reduce_gradients()
        self.postprocess_and_apply()
        return out
