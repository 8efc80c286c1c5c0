"""ASR regularisers of AIR-ASR as one fused per-image kernel (fwd) + one (bwd).

Mirrors ``air/air_number_bbox_location.py``: entropy ``:645-681``, marginal / min-element count
penalties ``:970-1015``, size window ``:1016-1027``, out-of-canvas / pairwise size / pairwise overlap
``:1029-1069``; they enter the loss as ``mean_b(elbo + per_image) + margin`` (``:1078-1079``).
"""
from __future__ import annotations

import ctypes
from dataclasses import dataclass, field
from typing import Optional, Sequence

import torch

from . import _lib
from .transformer import _need_cuda, _stream

COMPONENT_NAMES = ("pr_num", "num_min_KL", "area_loss", "out_loss", "size_loss", "over_loss")


@dataclass
class AsrRegulariser:
    """Hyper-parameters in the reference's vocabulary (train_air_pr.py:40-61,:177-212)."""
    canvas_size: float
    max_steps: int
    constrains_num: Sequence[int] = field(default_factory=list)   # digits of -dn
    constrains_num_gamma: float = 0.0            # -gn
    constrains_margin_gamma: float = 0.0         # -gm
    constrains_num_element_gamma: float = 0.0    # -gne
    constrains_bbox_gamma: float = 0.0           # -gb
    constrains_sharesize_gamma: float = 0.0      # -gs
    constrains_area_gamma: float = 0.0           # -ga
    constrains_area_minmax: Sequence[float] = (0.0, 0.0)

    def c_config(self) -> _lib.AsrConfig:
        c = _lib.AsrConfig()
        c.canvas_size = float(self.canvas_size)
        c.max_steps = int(self.max_steps)
        counts = list(self.constrains_num)
        if len(counts) > _lib.MOG_ASR_MAX_COUNTS:
            raise ValueError(f"at most {_lib.MOG_ASR_MAX_COUNTS} counts supported")
        c.num_counts = len(counts)
        for i, v in enumerate(counts):
            c.counts[i] = int(v)
        c.gamma_num = float(self.constrains_num_gamma)
        c.gamma_margin = float(self.constrains_margin_gamma)
        c.gamma_elem = float(self.constrains_num_element_gamma)
        c.gamma_bbox = float(self.constrains_bbox_gamma or 0.0)
        c.gamma_size = float(self.constrains_sharesize_gamma or 0.0)
        c.gamma_area = float(self.constrains_area_gamma)
        c.size_min = float(self.constrains_area_minmax[0])
        c.size_max = float(self.constrains_area_minmax[1])
        return c

    def __call__(self, log_odds, shifts, scales, **kw):
        return asr_regularisers(self, log_odds, shifts, scales, **kw)


class _AsrReg(torch.autograd.Function):
    @staticmethod
    def forward(ctx, log_odds, shifts, scales, cfg, psum, inv_B, want_components):
        L = _lib.load()
        B, T = log_odds.shape
        dev = log_odds.device
        per_image = torch.empty(B, dtype=torch.float32, device=dev)
        margin = torch.empty(1, dtype=torch.float32, device=dev)
        comps = torch.empty((B, _lib.MOG_ASR_NUM_COMPONENTS), dtype=torch.float32, device=dev) if want_components else None
        with torch.cuda.device(dev):
            _lib.check(L.mog_asr_reg_forward(log_odds.data_ptr(), shifts.data_ptr(), scales.data_ptr(),
                                             psum.data_ptr() if psum is not None else None, inv_B, B, T,
                                             ctypes.byref(cfg), per_image.data_ptr(),
                                             comps.data_ptr() if comps is not None else None, margin.data_ptr(),
                                             _stream(log_odds)), "mog_asr_reg_forward")
        ctx.save_for_backward(log_odds, shifts, scales, psum)
        ctx.cfg, ctx.inv_B = cfg, inv_B
        if comps is not None:
            ctx.mark_non_differentiable(comps)
            return per_image, margin.reshape(()), comps
        return per_image, margin.reshape(()), torch.empty(0, device=dev)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g_per_image, g_margin, _g_comps):
        log_odds, shifts, scales, psum = ctx.saved_tensors
        L = _lib.load()
        B, T = log_odds.shape
        d_lo, d_sh, d_sc = torch.empty_like(log_odds), torch.empty_like(shifts), torch.empty_like(scales)
        g_per_image = g_per_image.to(torch.float32).contiguous()
        g_margin = g_margin.to(torch.float32).reshape(1).contiguous()
        with torch.cuda.device(log_odds.device):
            _lib.check(L.mog_asr_reg_backward(log_odds.data_ptr(), shifts.data_ptr(), scales.data_ptr(),
                                              psum.data_ptr() if psum is not None else None, ctx.inv_B,
                                              g_per_image.data_ptr(), g_margin.data_ptr(), B, T, ctypes.byref(ctx.cfg),
                                              d_lo.data_ptr(), d_sh.data_ptr(), d_sc.data_ptr(), _stream(log_odds)),
                       "mog_asr_reg_backward")
        return d_lo, d_sh, d_sc, None, None, None, None


def asr_regularisers(cfg: AsrRegulariser, log_odds, shifts, scales, *, process_group=None,
                     global_batch: Optional[int] = None, want_components: bool = True):
    """Returns ``(per_image [B], margin scalar, components [B,6] or None)``.

    log_odds : ``[B, T]`` posterior z_pres log-odds of the executed steps (``z_pres_probs = sigmoid(.)``, :641-643)
    shifts   : ``[B, T, 2]`` ``rec_shifts`` (:923);  scales : ``[B, T]`` or ``[B, T, 1]`` ``rec_scales`` (:922)
    The marginal count penalty needs ``mean_b P[b,t]`` over the *global* batch (:982): with a
    ``process_group`` the per-rank column sums are all-reduced (one ``[T]`` float exchange) before use.
    """
    for t, n in ((log_odds, "log_odds"), (shifts, "shifts"), (scales, "scales")):
        _need_cuda(t, n)
    log_odds = log_odds.to(torch.float32).contiguous()
    B, T = log_odds.shape
    shifts = shifts.to(torch.float32).reshape(B, T, 2).contiguous()
    scales = scales.to(torch.float32).reshape(B, T).contiguous()
    c = cfg.c_config()
    psum = None
    nglobal = B if global_batch is None else int(global_batch)
    if c.gamma_margin > 1e-8:
        L = _lib.load()
        psum = torch.zeros(T, dtype=torch.float32, device=log_odds.device)
        with torch.cuda.device(log_odds.device):
            _lib.check(L.mog_asr_reg_colsum(log_odds.detach().data_ptr(), psum.data_ptr(), B, T, _stream(log_odds)),
                       "mog_asr_reg_colsum")
        if process_group is not None:
            import torch.distributed as dist
            dist.all_reduce(psum, group=process_group)
            if global_batch is None:
                nglobal = B * dist.get_world_size(process_group)
    per_image, margin, comps = _AsrReg.apply(log_odds, shifts, scales, c, psum, 1.0 / max(nglobal, 1), want_components)
    return per_image, margin, (comps if want_components else None)


class _AsrRegExecuted(torch.autograd.Function):
    """``_AsrReg`` over the executed steps only: ``psum`` holds ``2T`` floats, the second half the global active counts
    that give the trip count; ``steps`` is a non-differentiable 0-d int32 output."""

    @staticmethod
    def forward(ctx, log_odds, shifts, scales, cfg, psum, inv_B, want_components):
        L = _lib.load()
        B, T = log_odds.shape
        dev = log_odds.device
        per_image = torch.empty(B, dtype=torch.float32, device=dev)
        margin = torch.empty(1, dtype=torch.float32, device=dev)
        steps = torch.empty((), dtype=torch.int32, device=dev)
        comps = torch.empty((B, _lib.MOG_ASR_NUM_COMPONENTS), dtype=torch.float32, device=dev) if want_components else None
        with torch.cuda.device(dev):
            _lib.check(L.mog_asr_reg_forward_steps(log_odds.data_ptr(), shifts.data_ptr(), scales.data_ptr(), psum.data_ptr(),
                                                   inv_B, B, T, ctypes.byref(cfg), per_image.data_ptr(),
                                                   comps.data_ptr() if comps is not None else None, margin.data_ptr(),
                                                   steps.data_ptr(), _stream(log_odds)), "mog_asr_reg_forward_steps")
        ctx.save_for_backward(log_odds, shifts, scales, psum)
        ctx.cfg, ctx.inv_B = cfg, inv_B
        if comps is None:
            comps = torch.empty(0, device=dev)
        ctx.mark_non_differentiable(comps, steps)
        return per_image, margin.reshape(()), comps, steps

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g_per_image, g_margin, _g_comps, _g_steps):
        log_odds, shifts, scales, psum = ctx.saved_tensors
        L = _lib.load()
        B, T = log_odds.shape
        d_lo, d_sh, d_sc = torch.empty_like(log_odds), torch.empty_like(shifts), torch.empty_like(scales)
        g_per_image = g_per_image.to(torch.float32).contiguous()
        g_margin = g_margin.to(torch.float32).reshape(1).contiguous()
        with torch.cuda.device(log_odds.device):
            _lib.check(L.mog_asr_reg_backward_steps(log_odds.data_ptr(), shifts.data_ptr(), scales.data_ptr(), psum.data_ptr(),
                                                    ctx.inv_B, g_per_image.data_ptr(), g_margin.data_ptr(), B, T,
                                                    ctypes.byref(ctx.cfg), d_lo.data_ptr(), d_sh.data_ptr(), d_sc.data_ptr(),
                                                    _stream(log_odds)), "mog_asr_reg_backward_steps")
        return d_lo, d_sh, d_sc, None, None, None, None


def asr_regularisers_executed(cfg: AsrRegulariser, log_odds, shifts, scales, active, *, process_group=None,
                              global_batch: Optional[int] = None, want_components: bool = True):
    """The regularisers of the steps the reference loop executes (``while any(stop_sum < thr)``, :386-390), for a step
    that always runs ``T`` iterations.  Returns ``(per_image [B], margin scalar, components [B,6] or None, steps)``;
    ``steps`` is a 0-d int32 device tensor: ``1 + (first t <= T-2 with no active image after step t)``, or ``T``.

    Same arguments as ``asr_regularisers`` plus ``active`` ``[T, B]`` (bool or uint8): ``stop_sum < thr`` after each step.
    The trip count is that of the *global* batch: with a ``process_group`` the per-rank column sums and active counts are
    all-reduced in one ``[2T]`` float exchange.  Everything stays on the device (CUDA-graph capturable, no host read).
    The gradients of the columns ``t >= steps`` are exact zeros."""
    for t, n in ((log_odds, "log_odds"), (shifts, "shifts"), (scales, "scales"), (active, "active")):
        _need_cuda(t, n)
    log_odds = log_odds.to(torch.float32).contiguous()
    B, T = log_odds.shape
    shifts = shifts.to(torch.float32).reshape(B, T, 2).contiguous()
    scales = scales.to(torch.float32).reshape(B, T).contiguous()
    if tuple(active.shape) != (T, B) or active.dtype not in (torch.bool, torch.uint8):
        raise ValueError(f"active must be a [T, B] = [{T}, {B}] bool / uint8 tensor, got {tuple(active.shape)} {active.dtype}")
    active = active.detach().contiguous()
    c = cfg.c_config()
    L = _lib.load()
    psum = torch.zeros(2 * T, dtype=torch.float32, device=log_odds.device)
    with torch.cuda.device(log_odds.device):
        _lib.check(L.mog_asr_reg_colsum_steps(log_odds.detach().data_ptr(), active.data_ptr(), psum.data_ptr(), B, T,
                                              _stream(log_odds)), "mog_asr_reg_colsum_steps")
    nglobal = B if global_batch is None else int(global_batch)
    if process_group is not None:
        import torch.distributed as dist
        dist.all_reduce(psum, group=process_group)
        if global_batch is None:
            nglobal = B * dist.get_world_size(process_group)
    per_image, margin, comps, steps = _AsrRegExecuted.apply(log_odds, shifts, scales, c, psum, 1.0 / max(nglobal, 1),
                                                            want_components)
    return per_image, margin, (comps if want_components else None), steps
