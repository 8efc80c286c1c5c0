"""ORACLE (test infrastructure, NOT product code) -- the pixel-overlap placement of the dataset feeder
(``mog_synth_place_pixels``, ``DeviceMultiObjectDataset(mode="pixel")``), restated on the host.

The reference's rule for its non-"bbox" datasets (``/root/reference/multi_mnist.py:53-57,:180-182``): a position is
rejected only when the new object's pixels touch pixels already on the canvas.  Draws, attempts and restarts are those of
``synth_ref.place`` (same counter-based hash); candidates are evaluated with the C sampler oracle on ``synth_ref.box_theta``.
**Unpinned**: the reference's ``add_buffer`` cannot be read here, so the dilation by ``gap`` is this project's choice."""
import numpy as np

from . import stn_ref_c
from .synth_ref import box_theta, draw32, draw_int


def dilate(mask, gap):
    """``mask`` widened by ``gap`` pixels in Chebyshev distance (a (2 gap + 1)^2 square), clipped to the canvas"""
    if gap <= 0:
        return mask.copy()
    H, W = mask.shape
    out = np.zeros_like(mask)
    gy, gx = min(gap, H - 1), min(gap, W - 1)           # a wider shift leaves the canvas
    for dy in range(-gy, gy + 1):
        for dx in range(-gx, gx + 1):
            ys, yd = (slice(0, H - dy), slice(dy, H)) if dy >= 0 else (slice(-dy, H), slice(0, H + dy))
            xs, xd = (slice(0, W - dx), slice(dx, W)) if dx >= 0 else (slice(-dx, W), slice(0, W + dx))
            out[yd, xd] |= mask[ys, xs]
    return out


def place_pixels(sprites, seed, first_canvas, B, canvas, counts, size_min, size_max, gap=0, margin=0, share_size=False,
                 max_restarts=32, chunk=16):
    """``place`` with the reference's pixel-overlap rule (multi_mnist.py:53-57,:180-182) instead of a box test: a candidate
    is rejected when a pixel of its pasted layer (``paste``'s per-object value before the sum, >= 0.05) lies within
    Chebyshev distance ``gap`` of such a pixel of an object already placed.  Same draws, attempts and restarts as
    ``place``.  Candidates are evaluated with the C oracle (``stn_ref_c.forward`` of the sprite with ``box_theta``),
    ``chunk`` attempts per call; the first attempt that fits is taken."""
    sprites = np.asarray(sprites, np.float32)
    num_sprites = sprites.shape[0]
    G = max(1, max(counts))
    num = np.zeros(B, np.int32)
    pos, size, sprite = np.zeros((B, G, 2), np.int32), np.zeros((B, G, 2), np.int32), np.zeros((B, G), np.int32)
    for b in range(B):
        cid = first_canvas + b
        n = counts[draw_int(draw32(seed, cid, 0, 0, 0, 7), 0, len(counts))]
        placed = []
        for restart in range(max_restarts):
            placed = []
            occ = np.zeros((canvas, canvas), bool)                                                      # dilated occupancy
            shared = draw_int(draw32(seed, cid, restart, 0, 0, 1), size_min, size_max + 1)
            ok = True
            for i in range(n):
                w = shared if share_size else draw_int(draw32(seed, cid, restart, i, 0, 2), size_min, size_max + 1)
                sp = draw_int(draw32(seed, cid, restart, i, 0, 3), 0, num_sprites)
                span = canvas - w - 2 * margin + 1
                hit = None
                if span > 0:
                    for a0 in range(0, 100, chunk):
                        att = range(a0, min(100, a0 + chunk))
                        xy = np.array([[margin + draw_int(draw32(seed, cid, restart, i, a, 4), 0, span),
                                        margin + draw_int(draw32(seed, cid, restart, i, a, 5), 0, span)] for a in att], np.int32)
                        th = box_theta(xy, np.full_like(xy, w), canvas)
                        U = np.broadcast_to(sprites[sp][None, :, :, None], (len(att),) + sprites.shape[1:] + (1,))
                        masks = np.clip(stn_ref_c.forward(U, th, (canvas, canvas))[..., 0], 0.0, 1.0) >= 0.05
                        free = [k for k in range(len(att)) if not (masks[k] & occ).any()]
                        if free:
                            hit = (int(xy[free[0], 0]), int(xy[free[0], 1]), masks[free[0]])
                            break
                if hit is None:
                    ok = False
                    break
                x, y, m = hit
                occ |= dilate(m, gap)
                placed.append((x, y, w, sp))
            if ok:
                break
        num[b] = len(placed)
        for g, (x, y, w, sp) in enumerate(placed):
            pos[b, g], size[b, g], sprite[b, g] = (x, y), (w, w), sp
    return num, pos, size, sprite
