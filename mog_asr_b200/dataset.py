"""On-device synthetic Multi-MNIST / Multi-dSprites feeder: the in-memory replacement for the reference's generator +
TFRecord + ``shuffle_batch`` queue (``multi_mnist.py:90-301``, ``train_air_pr.py:144-147``).

Placement follows ``generate_multi_image`` (``multi_mnist.py:110-221``) and runs as one kernel (``mog_synth_place``;
``mode="pixel"``: ``mog_synth_place_pixels``, the reference's pixel-overlap rule ``:53-57,:180-182`` tested on the values
``paste`` will write); the pixels are then pasted by the sampler itself: every object is one write-direction
``transformer`` call of its sprite onto the canvas box (bilinear; the reference rescales with an order-5 spline, ``:144-153``), clipped to [0, 1],
values below 0.05 dropped (``:153-154``) and summed onto the canvas (``:200``).  With ``angles`` every object is also
rotated by an angle drawn from that set and labelled with its tight box (``:144-163``), under any of the three rules
(``mog_synth_place_rotated``; the paste then takes the theta the placement returns).  Canvases are a pure function of
``(seed, canvas index)``: any batch size, any rank split and any replay order give the same images.  Labels come in
the layout ``detection_metrics`` takes (positions, sizes, counts)."""
from __future__ import annotations

import ctypes
import math

import numpy as np
import torch

from . import _lib, synth
from .transformer import _need_cuda, _stream, transformer

MODES = {"bbox": 0, "disjoint": 1, "pixel": None}  # "pixel": mog_synth_place_pixels (no mode value of mog_synth_place)
PIXEL_MAX_CANVAS = 128  # MOG_SYNTH_PIXEL_MAX_CANVAS
MAX_ANGLES = 64  # MOG_SYNTH_MAX_ANGLES
ROTATED_MODES = {"bbox": 0, "disjoint": 1, "pixel": 2}  # the mode values of mog_synth_place_rotated


def dsprites_angles():
    """the 40 orientations of dSprites, whose shapes the reference bundles (``data/multi_dsprites/data.npz``): 40 values
    over the full circle, ``np.linspace(0, 360, 40)`` degrees with both ends included as in dSprites"""
    return tuple(float(a) for a in np.linspace(0.0, 360.0, 40))


def rotation_table(angles):
    """``[A, 2]`` float64 (cos, sin) of angles in degrees: the table ``mog_synth_place_rotated`` draws from"""
    return np.array([(math.cos(math.radians(a)), math.sin(math.radians(a))) for a in angles], np.float64).reshape(-1, 2)


def default_sprites(num=256, side=28, seed=0):
    """digit-like stroke sprites (MNIST cannot be downloaded here): ``[num, side, side]`` float32 in [0, 1]"""
    rng = np.random.default_rng(seed)
    return np.stack([synth._blob(rng, side) for _ in range(num)])


class DeviceMultiObjectDataset:
    def __init__(self, sprites, canvas_size=50, counts=(1, 3), size_range=(17, 23), gap=0, margin=0, mode="disjoint",
                 share_size=False, seed=0, device="cuda", angles=None):
        """``angles``: None, or a sequence of 1 to 64 angles in degrees (e.g. ``dsprites_angles()``).  Every object is then
        rotated by one of them, drawn uniformly, and labelled with its tight box; ``canvas_size <= 128`` in every mode."""
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("DeviceMultiObjectDataset needs a CUDA device: there is no CPU fallback")
        sp = torch.as_tensor(sprites, dtype=torch.float32)
        if sp.dim() != 3 or sp.shape[1] != sp.shape[2]:
            raise ValueError("sprites must be [num, side, side]")
        self.sprites = sp.to(self.device).contiguous()
        self.cs, self.counts = int(canvas_size), [int(c) for c in counts]
        self.size_min, self.size_max = int(size_range[0]), int(size_range[1])
        if self.size_min < 2 or self.size_max < self.size_min or self.size_max > self.cs:
            raise ValueError("size_range must satisfy 2 <= min <= max <= canvas_size")
        if mode not in MODES:
            raise ValueError(f"mode must be one of {sorted(MODES)}")
        self.gap, self.margin, self.mode, self.share_size, self.seed = int(gap), int(margin), mode, bool(share_size), int(seed)
        self.G = max(1, max(self.counts))
        self._counts_arr = (ctypes.c_int * len(self.counts))(*self.counts)
        self.angles = None if angles is None else tuple(float(a) for a in angles)
        if self.angles is not None:
            if not 1 <= len(self.angles) <= MAX_ANGLES:
                raise ValueError(f"angles must hold 1 to {MAX_ANGLES} values")
            if self.cs > PIXEL_MAX_CANVAS:
                raise ValueError(f"angles supports canvas_size <= {PIXEL_MAX_CANVAS}")
            rot = rotation_table(self.angles).reshape(-1)
            self._rot = (ctypes.c_double * rot.size)(*rot.tolist())
        elif mode == "pixel":
            if self.cs > PIXEL_MAX_CANVAS:
                raise ValueError(f"mode='pixel' supports canvas_size <= {PIXEL_MAX_CANVAS}")
            # the paste's theta entries t00 (per size) and t02 (per position and size), from box_theta itself, so that the
            # kernel's clash test sees exactly the values paste() writes
            p = torch.arange(self.cs, device=self.device)[:, None].expand(self.cs, self.size_max + 1)
            w = torch.arange(self.size_max + 1, device=self.device)[None, :].expand(self.cs, self.size_max + 1)
            th = self.box_theta(torch.stack([p, p], -1), torch.stack([w, w], -1), self.cs)      # [cs, size_max + 1, 6]
            self._box_scale = th[0, :, 0].contiguous()
            self._box_offset = th[:, :, 2].contiguous()

    # ---- placement (one launch) -----------------------------------------------------------------------------
    def place(self, first_canvas: int, B: int):
        """``(num, pos, size, sprite)``; with ``angles`` also ``theta [B, G, 6]``, the paste theta of every object"""
        i32 = lambda *s: torch.empty(*s, dtype=torch.int32, device=self.device)
        num, pos, size, sprite = i32(B), i32(B, self.G, 2), i32(B, self.G, 2), i32(B, self.G)
        L = _lib.load()
        with torch.cuda.device(self.device):
            if self.angles is not None:
                theta = torch.empty(B, self.G, 6, dtype=torch.float32, device=self.device)
                _lib.check(L.mog_synth_place_rotated(self.seed, int(first_canvas), B, self.cs, self.G, self._counts_arr, len(self.counts),
                                                     self.size_min, self.size_max, self.gap, self.margin, ROTATED_MODES[self.mode],
                                                     int(self.share_size), self.sprites.data_ptr(), int(self.sprites.shape[0]),
                                                     int(self.sprites.shape[1]), self._rot, len(self.angles), num.data_ptr(),
                                                     pos.data_ptr(), size.data_ptr(), sprite.data_ptr(), theta.data_ptr(), _stream(num)),
                           "mog_synth_place_rotated")
                return num, pos, size, sprite, theta
            if self.mode == "pixel":
                _lib.check(L.mog_synth_place_pixels(self.seed, int(first_canvas), B, self.cs, self.G, self._counts_arr, len(self.counts),
                                                    self.size_min, self.size_max, self.gap, self.margin, int(self.share_size),
                                                    self.sprites.data_ptr(), int(self.sprites.shape[0]), int(self.sprites.shape[1]),
                                                    self._box_scale.data_ptr(), self._box_offset.data_ptr(), num.data_ptr(),
                                                    pos.data_ptr(), size.data_ptr(), sprite.data_ptr(), _stream(num)),
                           "mog_synth_place_pixels")
                return num, pos, size, sprite
            _lib.check(L.mog_synth_place(self.seed, int(first_canvas), B, self.cs, self.G, self._counts_arr, len(self.counts),
                                         self.size_min, self.size_max, self.gap, self.margin, MODES[self.mode], int(self.share_size),
                                         int(self.sprites.shape[0]), num.data_ptr(), pos.data_ptr(), size.data_ptr(),
                                         sprite.data_ptr(), _stream(num)), "mog_synth_place")
        return num, pos, size, sprite

    # ---- paste: the sampler's write direction ---------------------------------------------------------------
    @staticmethod
    def box_theta(pos, size, canvas_size):
        """backward ST matrix that maps the sprite's [-1, 1] square onto canvas pixels [x, x+w-1] x [y, y+h-1];
        evaluated in float64 and rounded once, so host and device agree bit for bit"""
        p, s = pos.to(torch.float64), size.to(torch.float64)
        d = float(canvas_size - 1)
        sc = (s - 1.0) / d                                     # scale per axis
        c = -1.0 + (2.0 * p + s - 1.0) / d                      # centre per axis
        sc = torch.where(s > 0, sc, torch.ones_like(sc))       # unused slots: any finite matrix (masked out later)
        z = torch.zeros_like(sc[..., 0])
        th = torch.stack([1.0 / sc[..., 0], z, -c[..., 0] / sc[..., 0], z, 1.0 / sc[..., 1], -c[..., 1] / sc[..., 1]], -1)
        return th.to(torch.float32)

    def paste(self, num, pos, size, sprite, theta=None):
        """``theta``: the one ``place`` returns with ``angles`` (None: ``box_theta`` of the square boxes)"""
        B, G, cs = num.shape[0], self.G, self.cs
        U = self.sprites.index_select(0, sprite.reshape(-1).long()).unsqueeze(-1)                      # [B*G, D, D, 1]
        th = self.box_theta(pos, size, cs) if theta is None else theta
        v = transformer(U, th.reshape(B * G, 6), (cs, cs)).reshape(B, G, cs * cs)
        v = torch.clamp(v, 0.0, 1.0)                                                                    # :153
        live = (torch.arange(G, device=self.device)[None, :] < num[:, None])[:, :, None]
        return torch.where((v >= 0.05) & live, v, torch.zeros_like(v)).sum(1)                           # :154, :200

    def batch(self, index: int, batch_size: int, rank: int = 0, world: int = 1):
        """canvases ``[index*batch_size*world + rank*batch_size, ... + batch_size)`` of the infinite stream"""
        first = (int(index) * world + rank) * batch_size
        placed = self.place(first, batch_size)
        labels = dict(zip(("num", "pos", "size", "sprite", "theta"), placed))      # theta only with angles
        return dict(images=self.paste(*placed), **labels, first_canvas=first)

    def stream(self, batch_size: int, steps: int, rank: int = 0, world: int = 1, start: int = 0):
        """the training loop's ``shuffle_batch`` replacement: ``steps`` resident device batches, generated on demand"""
        for k in range(start, start + steps):
            yield self.batch(k, batch_size, rank, world)
