"""ORACLE (test infrastructure, NOT product code) -- rotated objects labelled with their tight boxes
(``mog_synth_place_rotated``, ``DeviceMultiObjectDataset(..., angles=...)``), restated on the host.

The reference rotates each object and re-crops it to its tight box, which becomes its label
(``/root/reference/multi_mnist.py:144-163``).  Draws, attempts and restarts are those of ``synth_ref.place`` (same
counter-based hash) plus the angle index, field 6.  Each object owns the square of side
``e = min(canvas, ceil(w (|cos| + |sin|)))`` that holds its rotated w-square; its paste theta is the header's fp64
expression.  Candidates are evaluated with the C sampler oracle on the full canvas.  **Unpinned**: scipy's order-5
``rotate`` is not reproduced (the paste is bilinear) and the angle set is the caller's."""
import math

import numpy as np

from . import stn_ref_c
from .synth_pixel_ref import dilate
from .synth_ref import boxes_clash, draw32, draw_int


def extent(w, c, s, canvas):
    """side of the square that holds a w-square rotated by (c, s)"""
    return min(canvas, math.ceil(w * (abs(c) + abs(s))))


def rotated_theta(c, s, w, e, x, y, canvas):
    """include/mogstn.h's paste theta of an object of size w, angle (c, s), whose e-square sits at (x, y): float64
    Python arithmetic (no FMA), each entry rounded to float32 once"""
    d = float(canvas - 1)
    sc = (w - 1.0) / d
    cx = -1.0 + (2.0 * x + e - 1.0) / d
    cy = -1.0 + (2.0 * y + e - 1.0) / d
    return np.array([c / sc, s / sc, -(c * cx + s * cy) / sc, (0.0 - s) / sc, c / sc, -(c * cy - s * cx) / sc], np.float32)


def masks_of(sprites, sp, theta, canvas):
    """``[n, canvas, canvas]`` bool: where the full-canvas forward of sprite ``sp`` with each theta, clipped to [0, 1],
    is >= 0.05 (the pixels ``paste`` keeps)"""
    theta = np.asarray(theta, np.float32).reshape(-1, 6)
    U = np.broadcast_to(np.asarray(sprites, np.float32)[sp][None, :, :, None], (theta.shape[0],) + sprites.shape[1:] + (1,))
    return np.clip(stn_ref_c.forward(U, theta, (canvas, canvas))[..., 0], 0.0, 1.0) >= 0.05


def tight_box(mask):
    """(x, y, w, h) of a non-empty mask's row and column extents"""
    rows, cols = np.flatnonzero(mask.any(1)), np.flatnonzero(mask.any(0))
    return int(cols[0]), int(rows[0]), int(cols[-1] - cols[0] + 1), int(rows[-1] - rows[0] + 1)


def place_rotated(sprites, rot, seed, first_canvas, B, canvas, counts, size_min, size_max, gap=0, margin=0, mode=2,
                  share_size=False, max_restarts=32, chunk=16):
    """``rot`` [A, 2] float64 (cos, sin).  mode 0 / 1: the tight box, widened by ``gap``, against the placed tight boxes
    with ``synth_ref.boxes_clash``; mode 2: the mask against the placed masks dilated by ``gap``
    (``synth_pixel_ref.place_pixels``).  An empty mask clashes with nothing and is labelled with its e-square.
    Returns ``num [B]``, ``pos`` / ``size [B, G, 2]`` (tight boxes), ``sprite [B, G]``, ``theta [B, G, 6]`` (unused slots
    0) and, for the tests, ``square [B, G, 3]``: each object's e-square (x, y, e)."""
    sprites = np.asarray(sprites, np.float32)
    rot = np.asarray(rot, np.float64).reshape(-1, 2)
    num_sprites = sprites.shape[0]
    G = max(1, max(counts))
    num = np.zeros(B, np.int32)
    pos, size, sprite = np.zeros((B, G, 2), np.int32), np.zeros((B, G, 2), np.int32), np.zeros((B, G), np.int32)
    theta, square = np.zeros((B, G, 6), np.float32), np.zeros((B, G, 3), np.int32)
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
                c, s = (float(v) for v in rot[draw_int(draw32(seed, cid, restart, i, 0, 6), 0, len(rot))])
                e = extent(w, c, s, canvas)
                span = canvas - e - 2 * margin + 1
                hit = None
                if span > 0:
                    for a0 in range(0, 100, chunk):
                        att = range(a0, min(100, a0 + chunk))
                        xy = [(margin + draw_int(draw32(seed, cid, restart, i, a, 4), 0, span),
                               margin + draw_int(draw32(seed, cid, restart, i, a, 5), 0, span)) for a in att]
                        th = np.stack([rotated_theta(c, s, w, e, x, y, canvas) for x, y in xy])
                        masks = masks_of(sprites, sp, th, canvas)
                        for k, (x, y) in enumerate(xy):
                            m = masks[k]
                            if not m.any():
                                box, empty = (x, y, e, e), True
                            else:
                                box, empty = tight_box(m), False
                                if mode == 2:
                                    if (m & occ).any():
                                        continue
                                elif any(boxes_clash(mode, *box, *q[0], gap) for q in placed if not q[1]):
                                    continue
                            hit = (box, empty, sp, th[k], m, (x, y, e))
                            break
                        if hit is not None:
                            break
                if hit is None:
                    ok = False
                    break
                if mode == 2:
                    occ |= dilate(hit[4], gap)
                placed.append(hit)
            if ok:
                break
        num[b] = len(placed)
        for g, (box, _empty, sp, th, _m, sq) in enumerate(placed):
            pos[b, g], size[b, g], sprite[b, g], theta[b, g], square[b, g] = box[:2], box[2:], sp, th, sq
    return num, pos, size, sprite, theta, square


def paste(sprites, canvas, num, sprite, theta):
    """``synth_ref.paste`` with the placement's theta instead of ``box_theta``"""
    B, G = sprite.shape
    U = np.asarray(sprites, np.float32)[sprite.reshape(-1)][..., None]
    v = stn_ref_c.forward(U, np.asarray(theta, np.float32).reshape(B * G, 6), (canvas, canvas)).reshape(B, G, canvas * canvas)
    v = np.clip(v, 0.0, 1.0)
    live = (np.arange(G)[None, :] < num[:, None])[:, :, None]
    out = np.zeros((B, canvas * canvas), np.float32)
    for g in range(G):                                      # same left-to-right sum as the device reduction over G <= 8
        out = out + np.where((v[:, g] >= 0.05) & live[:, g], v[:, g], np.float32(0))
    return out
