"""AIR-pPrior / AIR-ASR model (training graph) re-hosted in PyTorch.

Follows ``/root/reference/air/air_number_bbox_location.py`` (``AIRModel._create_model``, ``:384-1122``) op for
op; the places where the reference touches the hot path (and the canvas epilogue that follows it) go through an injectable ``ops`` object:

  * read    ``:511-542``  ``ops.transformer(images[B,cs,cs,1], theta_r, (ws, ws))``
  * write + composite ``:563-600,:718-727``  ``ops.write_composite(canvas, vae_recon, theta_w, z_pres, stop_sum, thr)``
  * ASR regularisers ``:645-681,:970-1069``  ``ops.asr(cfg, log_odds[B,T], shifts[B,T,2], scales[B,T,1], ...)``
  * reconstruction loss ``:945-968``  ``ops.recon_loss(images, canvas)`` (the epilogue right after the hot path)

``CudaOps`` (default) binds them to libmogstn's kernels.  The dense layers, LSTM cells and the elementwise
KL / Concrete math stay in PyTorch (cuBLAS GEMMs; SURVEY 2.1 marks them out of scope as kernels).

Random draws (TF's ``random_normal`` / ``random_uniform`` streams cannot be reproduced) come from a
``noise`` callback so that a step can be replayed with identical noise on another implementation.
"""
from __future__ import annotations

import contextlib
import math
import os
from dataclasses import dataclass, field
from typing import Callable, Optional, Sequence

import torch
import torch.nn as nn
import torch.nn.functional as F


@dataclass
class AIRConfig:
    """Keyword arguments of the reference ``AIRModel`` as ``train_air_pr.py:174-212`` passes them."""
    canvas_size: int = 50
    windows_size: int = 28
    max_steps: int = 6
    rnn_units: int = 256
    vae_latent_dimensions: int = 50
    vae_recognition_units: Sequence[int] = (512, 256)
    vae_generative_units: Sequence[int] = (256, 512)
    scale_hidden_units: int = 64
    shift_hidden_units: int = 64
    z_pres_hidden_units: int = 64
    scale_prior_mean: float = -1.0          # fix_scale_distribution=True (:74-76)
    scale_prior_variance: float = 0.05
    vae_prior_mean: float = 0.0
    vae_prior_variance: float = 1.0
    vae_likelihood_std: float = 0.0
    z_pres_temperature: float = 0.1         # -zt
    stopping_threshold: float = 0.9
    learning_rate: float = 1e-4
    gradient_clipping_norm: float = 1.0
    constrains_num: Sequence[int] = field(default_factory=lambda: [1, 3])   # digits of -dn
    constrains_num_gamma: float = 0.0            # -gn
    constrains_margin_gamma: float = 0.0         # -gm
    constrains_num_element_gamma: float = 0.0    # -gne
    constrains_bbox_gamma: float = 0.0           # -gb
    constrains_sharesize_gamma: float = 0.0      # -gs
    constrains_area_gamma: float = 0.0           # -ga
    constrains_area_minmax: Sequence[float] = (17.0, 23.0)
    fix_steps: Optional[int] = None              # the count when -dn has one digit (train_air_pr.py:212)
    always_max_steps: bool = False               # run max_steps iterations regardless of the `any` test (:386-390)
    stacked_kl: bool = True                      # evaluate the four KL terms once on [T,B,..] stacks after the loop
                                                 # (same elementwise math as the per-step form, 6x fewer launches)
    batched_tail: bool = True                    # with always_max_steps: everything that does not feed the next
                                                 # step's inference input (generative LSTM and prior heads, z_pres
                                                 # heads, VAE decoder, canvas writes) runs after the loop, the
                                                 # non-recurrent layers once over all T*B rows
    reference_trip_count: bool = False           # with always_max_steps: still max_steps iterations (capturable), but the
                                                 # ASR regularisers and `steps` cover only the iterations the reference
                                                 # loop executes, counted on the device (its loss and gradients)

    def __post_init__(self):
        if self.reference_trip_count and not self.always_max_steps:
            raise ValueError("reference_trip_count needs always_max_steps=True (the loop form already stops where the "
                             "reference does)")


def config_from_flags(data="mnist", dn="13", ds="", gn=0.0, gm=0.0, gne=0.0, gb=0.0, gs=0.0, ga=0.0, zt=0.1, **kw):
    """The derivations of ``train_air_pr.py:67-98,:204-212`` from its command-line flags."""
    counts = [int(c) for c in dn]
    if data.lower() == "mnist":
        cs, mm = 50, ((11, 15) if "bbox" in ds else (17, 23))
    else:
        cs, mm = 64, ((12, 15) if "bbox" in ds else (20, 25))
    return AIRConfig(canvas_size=cs, constrains_num=counts, constrains_num_gamma=gn, constrains_margin_gamma=gm,
                     constrains_num_element_gamma=gne, constrains_bbox_gamma=gb, constrains_sharesize_gamma=gs,
                     constrains_area_gamma=ga, constrains_area_minmax=mm, z_pres_temperature=zt,
                     fix_steps=counts[0] if len(counts) == 1 else None, **kw)


class CudaOps:
    """The hot-path operators bound to libmogstn (the product path).  ``fused_pointwise=False`` keeps the per-step
    elementwise math (sampling, theta construction, z_pres) in framework ops, written like the reference -- the
    kernels are still the sampler / composite / regulariser / loss ones; used to check the fused forms."""

    def __init__(self, process_group=None, global_batch=None, fused_pointwise=True, fused_heads=None):
        self.process_group, self.global_batch, self.fused_pointwise = process_group, global_batch, fused_pointwise
        self.fused_heads = fused_pointwise if fused_heads is None else fused_heads   # csrc/mog_air_head.cu

    def transformer(self, U, theta, out_size):
        from ..transformer import transformer
        return transformer(U, theta, out_size)

    def write_composite(self, canvas, window, theta, z_pres, stop_sum, threshold):
        from ..composite import write_composite
        return write_composite(canvas, window, theta, z_pres, stop_sum, threshold)

    def read_sxy(self, images4, inf_shift, inf_scale, out_size):
        """glimpse read with theta built in the kernel (``mog_asr_b200/sxy.py``); returns (window, shift, scale) -- the returned
        shift / scale go to ``write_composite_sxy`` so that their two gradients meet inside the read call's backward kernel"""
        if self.fused_pointwise:
            from ..sxy import read_glimpse_sxy
            return read_glimpse_sxy(images4, inf_shift, inf_scale, out_size)
        theta_r, _ = self.thetas(inf_shift, inf_scale)
        return self.transformer(images4, theta_r, out_size), inf_shift, inf_scale

    def write_composite_sxy(self, canvas, window, shift, scale, z_pres, stop_sum, threshold):
        if self.fused_pointwise:
            from ..sxy import write_composite_sxy
            return write_composite_sxy(canvas, window, shift, scale, z_pres, stop_sum, threshold)
        _, theta_w = self.thetas(shift, scale)
        return self.write_composite(canvas, window, theta_w, z_pres, stop_sum, threshold)

    def recon_loss(self, images, canvas):
        from ..recon import reconstruction_loss
        return reconstruction_loss(canvas, images)[0]

    # per-step elementwise math (csrc/mog_air.cu)
    def gauss_sample(self, mean, logvar, eps, act=None):
        if self.fused_pointwise:
            from .fused import gauss_sample
            return gauss_sample(mean, logvar, eps, act)
        latent = mean + eps * torch.sqrt(torch.exp(logvar))                                   # :180-184
        return latent, (torch.tanh(latent) if act == "tanh" else torch.sigmoid(latent) if act == "sigmoid" else None)

    def thetas(self, inf_shift, inf_scale):
        if self.fused_pointwise:
            from .fused import thetas
            return thetas(inf_shift, inf_scale)
        s, x, y = inf_scale[:, 0], inf_shift[:, 0], inf_shift[:, 1]
        zero = torch.zeros_like(s)
        return (torch.stack([s, zero, x, zero, s, y], 1),                                     # :511-531
                torch.stack([1.0 / s, zero, -x / s, zero, 1.0 / s, -y / s], 1))               # :563-584

    def kl_terms(self, stacks, cfg):
        """masked sum over steps of the four KL terms, one kernel each way; None = use the framework-op form"""
        if not self.fused_pointwise:
            return None
        from .fused import kl_terms
        return kl_terms(stacks, cfg.z_pres_temperature, cfg.scale_prior_mean, cfg.scale_prior_variance, cfg.vae_prior_mean,
                        cfg.vae_prior_variance)[0]

    @property
    def lstm_pointwise(self):
        if not self.fused_pointwise:
            return None
        from .fused import lstm_pointwise
        return lstm_pointwise

    def zpres(self, log_odds, u, stop_sum, temperature, threshold):
        if self.fused_pointwise:
            from .fused import zpres
            return zpres(log_odds, u, stop_sum, temperature, threshold)
        y_pre = (log_odds + torch.log(u + 10e-10) - torch.log(1.0 - u + 10e-10)) / temperature   # concrete.py:20-27
        z_pres = torch.sigmoid(y_pre)                                                         # :631
        stop_new = stop_sum + (1.0 - z_pres)                                                  # :712
        return y_pre, z_pres, stop_new, stop_sum < threshold, stop_new < threshold

    def asr(self, cfg: AIRConfig, log_odds, shifts, scales, active=None):
        """``active`` ``[T, B]`` given: the regularisers of the executed steps only, and their count as a 4th result"""
        from ..asr import AsrRegulariser, asr_regularisers, asr_regularisers_executed
        reg = AsrRegulariser(
            canvas_size=cfg.canvas_size, max_steps=cfg.max_steps, constrains_num=list(cfg.constrains_num),
            constrains_num_gamma=cfg.constrains_num_gamma, constrains_margin_gamma=cfg.constrains_margin_gamma,
            constrains_num_element_gamma=cfg.constrains_num_element_gamma, constrains_bbox_gamma=cfg.constrains_bbox_gamma,
            constrains_sharesize_gamma=cfg.constrains_sharesize_gamma, constrains_area_gamma=cfg.constrains_area_gamma,
            constrains_area_minmax=cfg.constrains_area_minmax)
        if active is not None:
            return asr_regularisers_executed(reg, log_odds, shifts, scales, active, process_group=self.process_group,
                                             global_batch=self.global_batch)
        return asr_regularisers(reg, log_odds, shifts, scales, process_group=self.process_group,
                                global_batch=self.global_batch)


class _DeferredAffine(torch.autograd.Function):
    """``y = base + x @ w`` (``w`` is ``[in, out]``; ``base`` is a bias vector or a per-row tensor) whose backward
    returns only ``dx`` (and ``dbase`` when ``base`` is a tensor with rows) and stashes ``(x, dy)``: the weight /
    bias gradients of a layer that is applied once per loop iteration are then formed by ONE GEMM over the
    concatenated rows of all iterations (``flush``) instead of one GEMM + one reduction + two accumulations per
    iteration.  Same sums, associated differently."""

    @staticmethod
    def forward(ctx, x, w, base, stash, base_is_bias):
        ctx.save_for_backward(x, w)
        ctx.stash, ctx.base_is_bias = stash, base_is_bias or base is None
        return torch.mm(x, w) if base is None else torch.addmm(base, x, w)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, dy):
        x, w = ctx.saved_tensors
        ctx.stash.append((x, dy))
        return dy @ w.t(), None, (None if ctx.base_is_bias else dy), None, None


class _StepAffine:
    """mixin: owns the stash of a layer that is applied once per loop iteration"""

    def _init_defer(self):
        self._stash, self.defer = [], False

    def _affine(self, x, w_in_out, bias, base=None):
        """x @ w + (base if given else bias); weight/bias gradients deferred when ``self.defer``."""
        if not (self.defer and torch.is_grad_enabled()):
            return torch.addmm(bias if base is None else base, x, w_in_out)
        return _DeferredAffine.apply(x, w_in_out, bias if base is None else base, self._stash, base is None)

    def flush(self, weight_grad_in_out, bias_grad, bias_from_stash=True):
        """accumulate the deferred gradients into the given .grad views and clear the stash"""
        if not self._stash:
            return
        with torch.no_grad():
            X = torch.cat([x.detach() for x, _ in self._stash], 0)
            DY = torch.cat([dy.detach() for _, dy in self._stash], 0)
            weight_grad_in_out.addmm_(X.t(), DY)
            if bias_from_stash and bias_grad is not None:
                bias_grad.addmv_(DY.t(), DY.new_ones(DY.shape[0]))      # column sums, accumulated in place
        self._stash.clear()


class StepLinear(nn.Module, _StepAffine):
    """``tf.layers.dense`` / ``layers.fully_connected`` (glorot-uniform kernel, zero bias) with deferrable weight
    gradients; parameters keep the nn.Linear layout (``weight [out, in]``, ``bias [out]``)."""

    def __init__(self, i, o):
        super().__init__()
        self.weight = nn.Parameter(torch.empty(o, i))
        self.bias = nn.Parameter(torch.zeros(o))
        nn.init.xavier_uniform_(self.weight)
        self._init_defer()
        self.fuse = False        # set by AIRModel when its ops object offers the fused epilogues

    def forward(self, x, act=None):
        """``act(x W^T + b)`` with ``act`` in None / 'relu' / 'softplus' / 'sigmoid'"""
        if self.fuse and self.defer and x.is_cuda and x.dtype == torch.float32 and torch.is_grad_enabled():
            from .fused import linear_act                      # library GEMM + one bias/activation kernel each way
            return linear_act(self, x, act)
        y = self._affine(x, self.weight.t(), self.bias)
        return y if act is None else {"relu": F.relu, "softplus": F.softplus, "sigmoid": torch.sigmoid}[act](y)

    def flush_grads(self):
        self.flush(self.weight.grad.t(), self.bias.grad)


class LSTMCellTF(nn.Module, _StepAffine):
    """``tf.nn.rnn_cell.LSTMCell(units)`` (:865-872): one kernel ``[in+units, 4*units]``, gate order i, j, f, o,
    ``forget_bias = 1.0`` added at run time, glorot-uniform kernel, zero bias  [TF-1.12 defaults]."""

    def __init__(self, input_size: int, units: int):
        super().__init__()
        self.units = units
        self.kernel = nn.Parameter(torch.empty(input_size + units, 4 * units))
        self.bias = nn.Parameter(torch.zeros(4 * units))
        nn.init.xavier_uniform_(self.kernel)
        self._init_defer()
        self._static_width = 0

    def flush_grads(self):
        # with a static block the bias gradient flows through static_gates (ordinary autograd), not the stash
        self.flush(self.kernel.grad[self._static_width:], self.bias.grad, bias_from_stash=(self._static_width == 0))

    def forward(self, x, state, static_gates=None, static_width=0, pointwise=None):
        """``static_gates`` = ``x_static @ kernel[:static_width]`` for a leading block of the input that does not
        change between steps (the flattened image, ``:416-419``): it is computed once per training step instead of
        once per loop iteration -- the same sum, associated differently -- and ``x`` then holds only the rest."""
        c, h = state
        self._static_width = static_width if static_gates is not None else 0
        xh = h if x.shape[1] == 0 else torch.cat([x, h], 1)
        if static_gates is not None and pointwise is not None and self.defer and torch.is_grad_enabled():
            # the static part (which carries the bias) is added inside the gate kernel: plain GEMM, no accumulate-into-a-copy
            dyn = _DeferredAffine.apply(xh, self.kernel[static_width:], None, self._stash, True)
            c2, h2 = pointwise(dyn, c, static_gates)
            return h2, (c2, h2)
        if static_gates is None:
            gates = self._affine(xh, self.kernel, self.bias)
        else:
            gates = self._affine(xh, self.kernel[static_width:], self.bias, base=static_gates)
        if pointwise is not None:
            c2, h2 = pointwise(gates, c)
        else:
            i, j, f, o = gates.chunk(4, 1)
            c2 = torch.sigmoid(f + 1.0) * c + torch.sigmoid(i) * torch.tanh(j)
            h2 = torch.sigmoid(o) * torch.tanh(c2)
        return h2, (c2, h2)

    def static_part(self, x_static):
        """bias + x_static @ kernel[:width]  (one GEMM per training step for the image block)"""
        w = x_static.shape[1]
        return torch.addmm(self.bias, x_static, self.kernel[:w]), w


def _dense(i, o):
    """``tf.layers.dense`` / ``layers.fully_connected`` defaults: glorot-uniform kernel, zero bias."""
    return StepLinear(i, o)


class _MeanVar(nn.Module):
    """Two 2-layer heads (mean, log-variance) of the shift / scale blocks (:424-460, :472-481)."""

    def __init__(self, in_dim, hidden, out_dim, skip_dim=0):
        super().__init__()
        self.hm, self.m = _dense(in_dim + skip_dim, hidden), _dense(hidden + skip_dim, out_dim)
        self.hv, self.v = _dense(in_dim + skip_dim, hidden), _dense(hidden + skip_dim, out_dim)
        self.in_dim, self.skip_dim = in_dim, skip_dim
        self._w1cat, self._head_stash = None, []

    def forward(self, x, skip=None):
        if skip is None:
            return self.m(self.hm(x, "relu")), self.v(self.hv(x, "relu"))
        xs = torch.cat([x, skip], -1)                       # shared by the mean and the log-variance branch
        mean = self.m(torch.cat([self.hm(xs, "relu"), skip], -1))
        logvar = self.v(torch.cat([self.hv(xs, "relu"), skip], -1))
        return mean, logvar

    # ---- fused form (csrc/mog_air_head.cu): one library GEMM + one kernel each way ----------------------------------
    def fusable(self, ops, x):
        # (only inside a training step: the concatenated first-layer weight is rebuilt by prepare() at the start of every
        #  differentiated forward pass and would be stale in a later no-grad evaluation)
        return (getattr(ops, "fused_heads", False) and self.hm.defer and torch.is_grad_enabled() and x.is_cuda
                and x.dtype == torch.float32 and self.hm.weight.shape[0] in (16, 32, 64, 128) and self.m.weight.shape[0] <= 2
                and self.skip_dim <= 2)

    def prepare(self):
        """[W1m | W1v] without the skip columns, rebuilt once per training step (the weights change every step)"""
        with torch.no_grad():
            self._w1cat = torch.cat([self.hm.weight[:, :self.in_dim], self.hv.weight[:, :self.in_dim]], 0)   # [2h, K]

    def sample(self, ops, x, eps, act, skip=None):
        """``(mean, logvar, latent, squashed)``: heads + reparameterised sample (:424-436 / :439-459)"""
        if self._w1cat is not None and self.fusable(ops, x):
            from .fused import fused_head
            return fused_head(self, x, skip, eps, act)
        mean, logvar = self(x, skip)
        latent, squashed = ops.gauss_sample(mean, logvar, eps, act)
        return mean, logvar, latent, squashed

    def flush_head(self):
        """first-layer weight / bias gradients from the rows stashed by the fused backward (one GEMM per head per step)"""
        if not self._head_stash:
            return
        with torch.no_grad():
            K, h = self.in_dim, self.hm.weight.shape[0]
            X = torch.cat([x for x, _, _ in self._head_stash], 0)
            D = torch.cat([d for _, _, d in self._head_stash], 0)
            dW = torch.mm(D.t(), X)                                                     # [2h, K]
            self.hm.weight.grad[:, :K] += dW[:h]
            self.hv.weight.grad[:, :K] += dW[h:]
            if self.skip_dim:
                Sk = torch.cat([s for _, s, _ in self._head_stash], 0)
                dWs = torch.mm(D.t(), Sk)                                               # [2h, S]
                self.hm.weight.grad[:, K:] += dWs[:h]
                self.hv.weight.grad[:, K:] += dWs[h:]
            db = D.sum(0)
            self.hm.bias.grad += db[:h]
            self.hv.bias.grad += db[h:]
        self._head_stash.clear()


class _GaussPair:
    """mean / log-variance layers that share their input and feed one sample (vae.py:21-31): evaluated as one GEMM on the
    concatenated weights plus one kernel; their gradients come from the stashed ``(x, dpre)`` rows at flush time."""

    def __init__(self, mean_layer, logvar_layer):
        self.mean_layer, self.logvar_layer, self.wcat, self.stash = mean_layer, logvar_layer, None, []

    def usable(self, x):
        return (self.wcat is not None and self.mean_layer.fuse and self.mean_layer.defer and x.is_cuda and x.dtype == torch.float32
                and torch.is_grad_enabled())

    def prepare(self):
        with torch.no_grad():
            self.wcat = torch.cat([self.mean_layer.weight, self.logvar_layer.weight], 0)      # [2L, in]

    def reset(self):
        self.wcat = None
        self.stash.clear()

    def flush(self):
        if not self.stash:
            return
        with torch.no_grad():
            Ld = self.mean_layer.weight.shape[0]
            X = torch.cat([x for x, _ in self.stash], 0)
            D = torch.cat([d for _, d in self.stash], 0)
            dW = torch.mm(D.t(), X)
            self.mean_layer.weight.grad += dW[:Ld]
            self.logvar_layer.weight.grad += dW[Ld:]
            db = D.sum(0)
            self.mean_layer.bias.grad += db[:Ld]
            self.logvar_layer.bias.grad += db[Ld:]
        self.stash.clear()


class AIRModel(nn.Module):
    """Training graph of the reference ``AIRModel`` (``train=True``)."""

    def __init__(self, cfg: AIRConfig, ops=None):
        super().__init__()
        self.cfg, self.ops = cfg, (ops if ops is not None else CudaOps())
        H, L, cs2, ws2 = cfg.rnn_units, cfg.vae_latent_dimensions, cfg.canvas_size ** 2, cfg.windows_size ** 2
        self.infer_cell = LSTMCellTF(cs2 + L + 3, H)                        # :413-422
        self.inf_shift = _MeanVar(H, cfg.shift_hidden_units, 2)             # :424-437
        self.inf_scale = _MeanVar(H, cfg.scale_hidden_units, 1, skip_dim=2)  # :439-460
        self.gen_cell = LSTMCellTF(L + 3, H)                                # :465-470
        self.gen_shift = _MeanVar(H, cfg.shift_hidden_units, 2)             # :472-481
        r, gdim = list(cfg.vae_recognition_units), list(cfg.vae_generative_units)
        self.vae_rec = nn.ModuleList([_dense(a, b) for a, b in zip([ws2] + r[:-1], r)])          # vae.py:16-19
        self.vae_rec_mean, self.vae_rec_logvar = _dense(r[-1], L), _dense(r[-1], L)              # vae.py:21-26
        self.vae_gen = nn.ModuleList([_dense(a, b) for a, b in zip([L] + gdim[:-1], gdim)])      # vae.py:34-37
        self.vae_gen_mean = _dense(gdim[-1], ws2)                                                # vae.py:39-41
        if cfg.fix_steps is None:
            self.z_prior_h, self.z_prior = _dense(H, cfg.z_pres_hidden_units), _dense(cfg.z_pres_hidden_units, 1)  # :609-615
        self.z_post_h, self.z_post = _dense(H, cfg.z_pres_hidden_units), _dense(cfg.z_pres_hidden_units, 1)        # :620-623
        for m in self.modules():
            if isinstance(m, StepLinear):
                m.fuse = bool(getattr(self.ops, "fused_heads", False))
        self._vae_pair = _GaussPair(self.vae_rec_mean, self.vae_rec_logvar)

    # ---- parallel branches of the captured step -------------------------------------------------------------------
    # Inside a CUDA-graph capture independent chains of small kernels are recorded on side streams that fork from and
    # rejoin the capture stream: they become parallel branches of the graph (the step is a dependent chain of ~650 small
    # kernels; what bounds it at 512 images per GPU is the chain's length, not the work).  Autograd runs every node's
    # backward on the stream of its forward, so the backward pass forks the same way.  Outside a capture (eager mode) the
    # code runs on one stream: the caching allocator's cross-stream lifetime rules are not worth it there.
    def _branch_streams(self, device, n, what="gen"):
        mode = os.environ.get("MOG_AIR_STREAMS", "1")           # "0" off, "1" on, "gen" / "flush": one of the two uses only (experiments)
        if not (device.type == "cuda" and mode in ("1", what) and torch.cuda.is_current_stream_capturing()):
            return None
        pool = self.__dict__.setdefault("_side_streams", {})
        key = (device.index, n)
        if key not in pool:
            pool[key] = [torch.cuda.Stream(device) for _ in range(n)]
        return pool[key]

    # ---- deferred weight gradients (see _DeferredAffine) ------------------------------------------------------
    def set_deferred_weight_grads(self, on: bool):
        for m in self.modules():
            if isinstance(m, _StepAffine):
                m.defer = bool(on)
                m._stash.clear()
            if isinstance(m, _MeanVar):
                m._head_stash.clear()
                m._w1cat = None
        self._vae_pair.reset()

    def flush_weight_grads(self):
        jobs = []
        for m in self.modules():
            if isinstance(m, _StepAffine):
                jobs.append(m.flush_grads)
            if isinstance(m, _MeanVar):
                jobs.append(m.flush_head)
        jobs.append(self._vae_pair.flush)
        dev = next(self.parameters()).device
        side = self._branch_streams(dev, 3, "flush")
        if side is None:
            for j in jobs:
                j()
            return
        # every flush writes its own layer's .grad: independent GEMMs, dealt out over the capture stream and three branches.
        # The stashed rows were allocated on other streams than the one that reads them here: they are kept alive until the
        # branches have rejoined, so that the allocator cannot hand their memory to a kernel that is not ordered after the read.
        keep = []
        for m in self.modules():
            if isinstance(m, _StepAffine):
                keep.extend(m._stash)
            if isinstance(m, _MeanVar):
                keep.extend(m._head_stash)
        keep.extend(self._vae_pair.stash)
        main = torch.cuda.current_stream(dev)
        for st in side:
            st.wait_stream(main)
        lanes = [main] + side
        for k, j in enumerate(jobs):
            with torch.cuda.stream(lanes[k % len(lanes)]):
                j()
        for st in side:
            main.wait_stream(st)
        del keep

    # ---- pieces -------------------------------------------------------------------------------------------
    def _encode(self, window, eps):
        """recognition half of air/vae.py:5-31: softplus layers, mean / log-variance, sample"""
        x = window
        for l in self.vae_rec:
            x = l(x, "softplus")
        if self._vae_pair.usable(x):
            from .fused import linear_gauss
            return linear_gauss(self._vae_pair, x, eps)
        mean, logvar = self.vae_rec_mean(x), self.vae_rec_logvar(x)
        latent, _ = self.ops.gauss_sample(mean, logvar, eps)                 # vae.py:28-31
        return mean, logvar, latent

    def _decode(self, latent):
        """generative half (vae.py:34-41); likelihood_std = 0 drops the second noise"""
        x = latent
        for l in self.vae_gen:
            x = l(x, "softplus")
        return self.vae_gen_mean(x, "sigmoid")

    def _vae(self, window, eps):
        """air/vae.py:5-48 (softplus hidden layers, sigmoid output)"""
        mean, logvar, latent = self._encode(window, eps)
        return self._decode(latent), mean, logvar, latent

    @staticmethod
    def _concrete_kl(y, prior_lo, post_lo, temp, eps=10e-10):
        """air/concrete.py:30-64 with prior temperature == posterior temperature (:690-696)."""
        def logp(lo):
            lse = torch.logsumexp(torch.stack([torch.zeros_like(y), -y * temp + lo]), 0)
            return math.log(temp + eps) - y * (temp + 1) + lo - 2.0 * lse
        return logp(post_lo) - logp(prior_lo)

    def _gaussian_kls(self, sc_mean, sc_lv, sh_mean, sh_lv, g_sh_mean, g_sh_lv, v_mean, v_lv):
        """:731-736 (scale, fixed prior), :750-755 (shift, learned prior), :769-774 (VAE latent); last axis summed."""
        cfg = self.cfg
        scale_kl = 0.5 * (math.log(cfg.scale_prior_variance) - sc_lv - 1.0 + torch.exp(sc_lv) / cfg.scale_prior_variance
                          + (sc_mean - cfg.scale_prior_mean) ** 2 / cfg.scale_prior_variance).sum(-1)
        g_sh_var = torch.exp(g_sh_lv)
        shift_kl = 0.5 * (g_sh_lv - sh_lv - 1.0 + torch.exp(sh_lv) / g_sh_var + (sh_mean - g_sh_mean) ** 2 / g_sh_var).sum(-1)
        vae_kl = 0.5 * (math.log(cfg.vae_prior_variance) - v_lv - 1.0 + torch.exp(v_lv) / cfg.vae_prior_variance
                        + (v_mean - cfg.vae_prior_mean) ** 2 / cfg.vae_prior_variance).sum(-1)
        return scale_kl, shift_kl, vae_kl

    # ---- the training graph ----------------------------------------------------------------------------------
    def forward(self, images, noise: Optional[Callable] = None, any_reduce: Optional[Callable] = None,
                global_batch: Optional[int] = None, recon_loss_fn: Optional[Callable] = None, train: bool = True):
        """images ``[B, cs*cs]`` in [0,1].  ``noise(kind, step, shape)`` supplies N(0,1) ('shift','scale','vae')
        or U(0,1) ('concrete') draws.  ``any_reduce(flag_tensor)`` makes the loop condition global across ranks.
        ``recon_loss_fn(images, clipped_canvas) -> [B]`` replaces the reference's cross-entropy (:954-959); it
        exists for tests only: the reference term has gradients of 1e10 wherever the canvas is exactly 0 under
        an object pixel, which amplifies fp32 rounding noise of *any* implementation beyond comparison.
        ``train=False`` is the reference's test model (``train_air_pr.py:170-171``): z_pres is rounded to 0/1 right after
        the sigmoid (:634-635), so the stopping sum, the counts and the canvas are those of hard decisions; run it under
        ``torch.no_grad()`` -- this is what feeds ``detection.evaluation``.
        Returns a dict with ``loss`` (differentiable) and the reference's log variables.
        With ``cfg.reference_trip_count`` every one of the ``max_steps`` iterations still runs, and ``z_pres_probs``,
        ``rec_shifts`` and ``rec_scales`` keep ``max_steps`` columns; ``steps`` is then a 0-d int32 device tensor, the
        iteration count of the reference loop, and the columns ``>= steps`` are not part of the reference's result (the
        loss, its gradients, ``components`` and ``margin`` leave them out)."""
        cfg = self.cfg
        dev, dt = images.device, images.dtype
        B = images.shape[0]
        cs, ws, thr, temp = cfg.canvas_size, cfg.windows_size, cfg.stopping_threshold, cfg.z_pres_temperature
        if noise is None:
            noise = lambda kind, step, shape: (torch.rand(shape, device=dev, dtype=dt) if kind == "concrete"
                                               else torch.randn(shape, device=dev, dtype=dt))
        H, L = cfg.rnn_units, cfg.vae_latent_dimensions
        z = lambda *s: torch.zeros(*s, device=dev, dtype=dt)
        if torch.is_grad_enabled():
            for head in (self.inf_shift, self.inf_scale):
                if head.fusable(self.ops, images):
                    head.prepare()
            if self.vae_rec_mean.fuse and self.vae_rec_mean.defer and images.is_cuda and images.dtype == torch.float32:
                self._vae_pair.prepare()
        if train and cfg.always_max_steps and cfg.batched_tail and cfg.stacked_kl:
            return self._forward_batched_tail(images, noise, global_batch, recon_loss_fn)
        stop_sum = z(B)
        inf_state, gen_state = (z(B, H), z(B, H)), (z(B, H), z(B, H))
        gen_prev_out, prev_latent, prev_ss = z(B, H), z(B, L), z(B, 3)
        canvas = z(B, cs, cs)
        kl = {k: [] for k in ("z_pres_kl", "scale_kl", "shift_kl", "vae_kl")}
        hist = {}
        act_list = []
        lo_list, sh_list, sc_list = [], [], []
        images4 = images.reshape(B, cs, cs, 1)
        # the image block of the inference LSTM input is the same at every step: its 2500x1024 GEMM runs once
        img_gates, img_w = self.infer_cell.static_part(images)

        lstm_pw = getattr(self.ops, "lstm_pointwise", None)   # fused gate math when the ops object offers it
        step = 0
        while step < cfg.max_steps:
            if not cfg.always_max_steps and step > 0:        # cond (:386-390); step 0 always runs (stop_sum = 0)
                flag = (stop_sum < thr).any()
                if any_reduce is not None:
                    flag = any_reduce(flag)
                if not bool(flag):
                    break
            prev = torch.cat([prev_latent, prev_ss], -1)   # input of both cells besides the image / the state
            out, inf_state = self.infer_cell(prev, inf_state, static_gates=img_gates, static_width=img_w,
                                             pointwise=lstm_pw)                                             # :413-422
            sh_mean, sh_lv, shift_latent, inf_shift = self.inf_shift.sample(self.ops, out, noise("shift", step, (B, 2)), "tanh")   # :424-435
            sc_mean, sc_lv, scale_latent, inf_scale = self.inf_scale.sample(self.ops, out, noise("scale", step, (B, 1)), "sigmoid",
                                                                            skip=shift_latent)                                # :439-458
            ss_latent = torch.cat([shift_latent, scale_latent], -1)                                         # :463
            gen_out, gen_state = self.gen_cell(prev, gen_state, pointwise=lstm_pw)                          # :465-470
            g_sh_mean, g_sh_lv = self.gen_shift(gen_out)                                                    # :472-481

            window, w_shift, w_scale = self.ops.read_sxy(images4, inf_shift, inf_scale, (ws, ws))           # :511-542 (theta_r in the kernel)
            window = window.reshape(B, ws, ws)
            recon, v_mean, v_lv, v_latent = self._vae(window.reshape(B, ws * ws), noise("vae", step, (B, L)))  # :544-553

            if cfg.fix_steps is not None:                                                                   # :604-608
                prior_lo = torch.full((B,), 100.0 if step < cfg.fix_steps else -100.0, device=dev, dtype=dt)
            else:
                prior_lo = self.z_prior(self.z_prior_h(gen_prev_out, "relu")).reshape(B)                     # :609-615
            post_lo = self.z_post(self.z_post_h(out, "relu")).reshape(B)                                     # :620-623
            if train:
                y_pre, z_pres, stop_sum, active_prev, active = self.ops.zpres(post_lo, noise("concrete", step, (B,)), stop_sum,
                                                                              temp, thr)     # concrete.py:20-27, :631, :698-712
            else:
                u = noise("concrete", step, (B,))
                y_pre = (post_lo + torch.log(u + 10e-10) - torch.log(1.0 - u + 10e-10)) / temp               # concrete.py:20-27
                z_pres = torch.round(torch.sigmoid(y_pre))                                                    # :631, :634-635
                active_prev = stop_sum < thr
                stop_sum = stop_sum + (1.0 - z_pres)                                                          # :712
                active = stop_sum < thr
            act_list.append(active)
            canvas = self.ops.write_composite_sxy(canvas, recon.reshape(B, ws, ws), w_shift, w_scale, z_pres, stop_sum, thr)  # :563-600,:722-727

            if cfg.stacked_kl:
                # the KL terms are elementwise functions of per-step tensors: keep those, evaluate after the loop
                for k, v in (("y_pre", y_pre), ("prior_lo", prior_lo), ("post_lo", post_lo), ("active_prev", active_prev),
                             ("active", active), ("sc_mean", sc_mean), ("sc_lv", sc_lv), ("sh_mean", sh_mean), ("sh_lv", sh_lv),
                             ("g_sh_mean", g_sh_mean), ("g_sh_lv", g_sh_lv), ("v_mean", v_mean), ("v_lv", v_lv)):
                    hist.setdefault(k, []).append(v)
            else:
                z_kl = self._concrete_kl(y_pre, prior_lo, post_lo, temp)                                    # :690-696
                kl["z_pres_kl"].append(torch.where(active_prev, z_kl, torch.zeros_like(z_kl)))
                scale_kl, shift_kl, vae_kl = self._gaussian_kls(sc_mean, sc_lv, sh_mean, sh_lv, g_sh_mean, g_sh_lv, v_mean, v_lv)
                for k, v in (("scale_kl", scale_kl), ("shift_kl", shift_kl), ("vae_kl", vae_kl)):
                    kl[k].append(torch.where(active, v, torch.zeros_like(v)))                               # masks use the NEW stop_sum
            lo_list.append(post_lo); sh_list.append(inf_shift); sc_list.append(inf_scale)
            gen_prev_out, prev_latent, prev_ss = gen_out, v_latent, ss_latent
            step += 1

        H_ = {k: torch.stack(v, 0) for k, v in hist.items()} if cfg.stacked_kl else None                   # [T, B, ...]
        return self._epilogue(images, canvas, act_list, H_, kl, torch.stack(lo_list, 1), torch.stack(sh_list, 1),
                              torch.stack(sc_list, 1), step, global_batch, recon_loss_fn)

    def _forward_batched_tail(self, images, noise, global_batch, recon_loss_fn):
        """Same graph as the loop in ``forward`` with a fixed trip count, evaluated in dependency order rather than
        in program order.  The next step's inference input is ``[image, previous VAE latent, previous shift/scale]``
        (:413-422), so only the inference LSTM, the shift/scale heads, the glimpse read and the VAE encoder are truly
        sequential.  The generative LSTM (:465-470) is a chain of its own; its input half, its prior heads
        (:472-481, :609-615), the z_pres heads (:620-623) and the VAE decoder (vae.py:34-41) have no recurrence at
        all and run once over all ``T*B`` rows; the Concrete / stopping-sum scan and the canvas writes follow in
        step order.  Same sums, same noise per (kind, step); GEMMs see ``T*B`` rows instead of ``B``."""
        cfg = self.cfg
        dev, dt = images.device, images.dtype
        B, T = images.shape[0], cfg.max_steps
        cs, ws, thr, temp = cfg.canvas_size, cfg.windows_size, cfg.stopping_threshold, cfg.z_pres_temperature
        H, L = cfg.rnn_units, cfg.vae_latent_dimensions
        z = lambda *s: torch.zeros(*s, device=dev, dtype=dt)
        lstm_pw = getattr(self.ops, "lstm_pointwise", None)
        images4 = images.reshape(B, cs, cs, 1)
        img_gates, img_w = self.infer_cell.static_part(images)

        # ---- the recurrence proper -------------------------------------------------------------------------
        inf_state = (z(B, H), z(B, H))
        prev_latent, prev_ss = z(B, L), z(B, 3)
        per = {k: [] for k in ("out", "prev", "latent", "w_sxy", "sc_mean", "sc_lv", "sh_mean", "sh_lv", "v_mean", "v_lv",
                               "shift", "scale")}
        for step in range(T):
            prev = torch.cat([prev_latent, prev_ss], -1)
            out, inf_state = self.infer_cell(prev, inf_state, static_gates=img_gates, static_width=img_w, pointwise=lstm_pw)
            sh_mean, sh_lv, shift_latent, inf_shift = self.inf_shift.sample(self.ops, out, noise("shift", step, (B, 2)), "tanh")
            sc_mean, sc_lv, scale_latent, inf_scale = self.inf_scale.sample(self.ops, out, noise("scale", step, (B, 1)), "sigmoid",
                                                                            skip=shift_latent)
            x, w_shift, w_scale = self.ops.read_sxy(images4, inf_shift, inf_scale, (ws, ws))   # theta_r built in the kernel
            x = x.reshape(B, ws * ws)                                                  # C = 1: a view, no select
            v_mean, v_lv, v_latent = self._encode(x, noise("vae", step, (B, L)))
            for k, v in (("out", out), ("prev", prev), ("latent", v_latent), ("w_sxy", (w_shift, w_scale)), ("sc_mean", sc_mean),
                         ("sc_lv", sc_lv), ("sh_mean", sh_mean), ("sh_lv", sh_lv), ("v_mean", v_mean), ("v_lv", v_lv),
                         ("shift", inf_shift), ("scale", inf_scale)):
                per[k].append(v)
            prev_latent, prev_ss = v_latent, torch.cat([shift_latent, scale_latent], -1)

        # ---- generative LSTM: input half for all steps at once, then its own chain ---------------------------
        # (a chain of its own: under graph capture it is a parallel branch beside the z_pres heads, the decoder, the
        #  Concrete scan and the canvas writes below; it is needed again only by the KL terms of the epilogue)
        side = self._branch_streams(dev, 1)
        main = torch.cuda.current_stream(dev) if side is not None else None
        if side is not None:
            side[0].wait_stream(main)
        with (torch.cuda.stream(side[0]) if side is not None else contextlib.nullcontext()):
            gen_static, gen_w = self.gen_cell.static_part(torch.cat(per["prev"], 0))
            gen_static = gen_static.reshape(T, B, 4 * H).unbind(0)   # (unbind, not [step]: one stack in the backward pass
            gen_state, gen_outs, none = (z(B, H), z(B, H)), [], z(B, 0)  #  instead of T zero-filled scatters that are then added)
            for step in range(T):
                g_out, gen_state = self.gen_cell(none, gen_state, static_gates=gen_static[step], static_width=gen_w, pointwise=lstm_pw)
                gen_outs.append(g_out)
            g_sh_mean, g_sh_lv = self.gen_shift(torch.cat(gen_outs, 0))                                            # :472-481
            if cfg.fix_steps is not None:                                                                        # :604-608
                prior_lo = torch.full((T, B), -100.0, device=dev, dtype=dt)
                prior_lo[:cfg.fix_steps] = 100.0
            else:
                gen_prev = torch.cat([z(B, H)] + gen_outs[:-1], 0)
                prior_lo = self.z_prior(self.z_prior_h(gen_prev, "relu")).reshape(T, B)                    # :609-615
        post_lo = self.z_post(self.z_post_h(torch.cat(per["out"], 0), "relu")).reshape(T, B)            # :620-623

        # ---- VAE decoder for all steps (vae.py:34-41) ----------------------------------------------------------
        recon = self._decode(torch.cat(per["latent"], 0)).reshape(T, B, ws, ws).unbind(0)

        # ---- Concrete / stopping-sum scan and the canvas writes, in step order -----------------------------------
        stop_sum, canvas = z(B), z(B, cs, cs)
        y_pre_l, act_prev_l, act_l = [], [], []
        post_lo_t = post_lo.unbind(0)
        for step in range(T):
            y_pre, z_pres, stop_sum, active_prev, active = self.ops.zpres(post_lo_t[step], noise("concrete", step, (B,)), stop_sum,
                                                                          temp, thr)
            canvas = self.ops.write_composite_sxy(canvas, recon[step], *per["w_sxy"][step], z_pres, stop_sum, thr)
            y_pre_l.append(y_pre); act_prev_l.append(active_prev); act_l.append(active)

        if side is not None:
            main.wait_stream(side[0])          # the generative branch rejoins before the KL terms
        st = lambda k: torch.stack(per[k], 0)
        H_ = dict(y_pre=torch.stack(y_pre_l, 0), prior_lo=prior_lo, post_lo=post_lo, active_prev=torch.stack(act_prev_l, 0),
                  active=torch.stack(act_l, 0), sc_mean=st("sc_mean"), sc_lv=st("sc_lv"), sh_mean=st("sh_mean"), sh_lv=st("sh_lv"),
                  g_sh_mean=g_sh_mean.reshape(T, B, 2), g_sh_lv=g_sh_lv.reshape(T, B, 2), v_mean=st("v_mean"), v_lv=st("v_lv"))
        return self._epilogue(images, canvas, act_l, H_, None, post_lo.t().contiguous(), torch.stack(per["shift"], 1),
                              torch.stack(per["scale"], 1), T, global_batch, recon_loss_fn)

    # ---- the generation graph --------------------------------------------------------------------------------
    @torch.no_grad()
    def generate(self, batch_size: int, noise: Optional[Callable] = None, device=None, dtype=None):
        """Samples from the generative model: the reference's ``_create_generation`` (``air_number_bbox_location.py:1124-1361``),
        the third model-math call site of the sampler (``:1249``), fetched by the trainer as ``generated_samples``
        (``train_air_pr.py:241,:389``).  Per step: generative LSTM on the previous step's latents (``:1151-1156``) -> learned
        shift prior, sampled (``:1157-1169``) -> the scale is drawn from the fixed prior but then REPLACED by the constant
        ``mean(constrains_area_minmax) / canvas_size`` (``:1199-1205``; the drawn latent still feeds the next step, ``:1209-1211``)
        -> a VAE prior sample decoded and binarised by a Bernoulli draw (``vae_generation(..., sample_from_mean=True)``,
        ``air/vae.py:51-86``) -> written onto the canvas with ``theta_w`` and the rounded Concrete ``z_pres`` of the learned (or
        fixed-count) prior (``:1225-1303``); the loop stops when every image has stopped (``:1131-1135``).
        ``noise(kind, step, shape)``: N(0,1) for 'shift' / 'scale' / 'vae', U(0,1) for 'concrete' and 'bernoulli'.
        Returns ``samples [B, cs, cs, 1]``, ``num`` (objects per image), ``thetas [B, steps, 2, 3]`` (the write transforms the
        reference hands to its bounding-box overlay) and ``steps``."""
        cfg = self.cfg
        p0 = next(self.parameters())
        dev, dt = device or p0.device, dtype or p0.dtype
        B = int(batch_size)
        cs, ws, thr, temp = cfg.canvas_size, cfg.windows_size, cfg.stopping_threshold, cfg.z_pres_temperature
        H, L = cfg.rnn_units, cfg.vae_latent_dimensions
        if noise is None:
            noise = lambda kind, step, shape: (torch.rand(shape, device=dev, dtype=dt) if kind in ("concrete", "bernoulli")
                                               else torch.randn(shape, device=dev, dtype=dt))
        z = lambda *s: torch.zeros(*s, device=dev, dtype=dt)
        stop_sum, gen_state = z(B), (z(B, H), z(B, H))
        gen_prev_out, prev_latent, prev_ss = z(B, H), z(B, L), z(B, 3)
        canvas, digits, thetas = z(B, cs, cs), torch.zeros(B, dtype=torch.int32, device=dev), []
        scale_value = float(sum(cfg.constrains_area_minmax)) / len(cfg.constrains_area_minmax) / cs        # :1203-1204
        scale = torch.full((B, 1), scale_value, device=dev, dtype=dt)
        step = 0
        while step < cfg.max_steps and bool((stop_sum < thr).any()):                                      # :1131-1135
            gen_out, gen_state = self.gen_cell(torch.cat([prev_latent, prev_ss], -1), gen_state)           # :1151-1156
            g_sh_mean, g_sh_lv = self.gen_shift(gen_out)                                                   # :1157-1166
            shift_latent = g_sh_mean + noise("shift", step, (B, 2)) * torch.sqrt(torch.exp(g_sh_lv))       # :1168
            shift = torch.tanh(shift_latent)                                                               # :1169
            scale_latent = cfg.scale_prior_mean + noise("scale", step, (B, 1)) * math.sqrt(cfg.scale_prior_variance)   # :1196-1200
            latent = cfg.vae_prior_mean + noise("vae", step, (B, L)) * math.sqrt(cfg.vae_prior_variance)   # vae.py:63-66
            mean = self._decode(latent)                                                                    # vae.py:68-81 (likelihood_std = 0)
            window = torch.relu(torch.sign(mean - noise("bernoulli", step, (B, ws * ws))))                 # vae.py:83-84
            _, theta_w = self.ops.thetas(shift, scale)                                                     # :1225-1246
            thetas.append(theta_w.reshape(B, 2, 3))
            if cfg.fix_steps is not None:                                                                  # :1261-1265
                prior_lo = torch.full((B,), 100.0 if step < cfg.fix_steps else -100.0, device=dev, dtype=dt)
            else:
                prior_lo = self.z_prior(self.z_prior_h(gen_prev_out, "relu")).reshape(B)                   # :1267-1272
            u = noise("concrete", step, (B,))
            y_pre = (prior_lo + torch.log(u + 10e-10) - torch.log(1.0 - u + 10e-10)) / temp                # concrete.py:20-27
            z_pres = torch.round(torch.sigmoid(y_pre))                                                     # :1281-1285
            stop_sum = stop_sum + (1.0 - z_pres)                                                           # :1291
            digits = digits + (stop_sum < thr).to(torch.int32)                                             # :1294-1295
            canvas = self.ops.write_composite(canvas, window.reshape(B, ws, ws), theta_w, z_pres, stop_sum, thr)   # :1249-1257,:1297-1303
            gen_prev_out, prev_latent, prev_ss = gen_out, latent, torch.cat([shift_latent, scale_latent], -1)
            step += 1
        return dict(samples=canvas.reshape(B, cs, cs, 1), num=digits, steps=step,
                    thetas=torch.stack(thetas, 1) if thetas else z(B, 0, 2, 3))

    def _epilogue(self, images, canvas, act_list, H_, kl, log_odds, shifts, scales, T, global_batch, recon_loss_fn):
        """everything after the loop: object counts, KL terms (:690-787,:930-935), reconstruction loss (:945-968),
        ASR regularisers (:645-681,:970-1069) and the loss (:1078-1079)"""
        cfg = self.cfg
        B = images.shape[0]
        cs, temp = cfg.canvas_size, cfg.z_pres_temperature
        active = torch.stack(act_list, 0)                                                                   # [T, B]
        digits = active.sum(0, dtype=torch.int32)                                                           # :715-716
        if cfg.stacked_kl:
            fused_kl = self.ops.kl_terms(H_, cfg) if hasattr(self.ops, "kl_terms") else None
        if cfg.stacked_kl and fused_kl is not None:
            elbo = fused_kl                                                                                 # :690-787,:930-935 fused
        elif cfg.stacked_kl:
            z_kl = self._concrete_kl(H_["y_pre"], H_["prior_lo"], H_["post_lo"], temp)
            scale_kl, shift_kl, vae_kl = self._gaussian_kls(H_["sc_mean"], H_["sc_lv"], H_["sh_mean"], H_["sh_lv"],
                                                            H_["g_sh_mean"], H_["g_sh_lv"], H_["v_mean"], H_["v_lv"])
            zero = torch.zeros_like(z_kl)
            elbo = (torch.where(H_["active_prev"], z_kl, zero)
                    + torch.where(H_["active"], scale_kl + shift_kl + vae_kl, zero)).sum(0)                 # :930-935
        else:
            elbo = sum(torch.stack(v, 1).sum(-1) for v in kl.values())                                      # :930-935
        canvas2 = canvas.reshape(B, cs * cs)
        recon_c = torch.clamp(canvas2.detach(), 0.0, 1.0)                                                   # :947-948 (logged)
        if recon_loss_fn is None:
            rec_loss = self.ops.recon_loss(images, canvas2)                                                 # :947-959 fused
        else:
            rec_loss = recon_loss_fn(images, torch.clamp(canvas2, 0.0, 1.0))
        elbo = elbo + rec_loss                                                                              # :968
        if cfg.reference_trip_count:
            # the regularisers of the iterations the reference loop executes (:386-390), trip count counted on the device
            per_image, margin, comps, T = self.ops.asr(cfg, log_odds, shifts, scales, active=active)
        else:
            per_image, margin, comps = self.ops.asr(cfg, log_odds, shifts, scales)                          # :645-681,:970-1069
        nglobal = B if global_batch is None else global_batch
        # loss = mean_b(elbo + pr_loss + num_element_min) + num_marginal_loss  (:1078-1079); under data
        # parallelism each rank holds sum_local / B_global and the gradient all-reduce restores the mean
        loss = (elbo + per_image).sum() / nglobal + margin
        return dict(loss=loss, elbo=elbo.detach(), recon=rec_loss.detach(), steps=T, rec_num_digits=digits,
                    margin=margin.detach(), per_image_reg=per_image.detach(), components=comps,
                    rec_scales=scales.detach(), rec_shifts=shifts.detach(), z_pres_probs=torch.sigmoid(log_odds).detach(),
                    reconstruction=recon_c)
