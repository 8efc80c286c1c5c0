"""Synthetic-dataset feeder, pixel-overlap placement (``mode="pixel"``, ``mog_synth_place_pixels``): the reference's rule
for its non-"bbox" datasets (multi_mnist.py:53-57,:180-182) -- objects may share box area but no pixel (within ``gap``).
Checked against oracle/synth_pixel_ref.place_pixels (same counter-based draws, candidates evaluated with the C sampler oracle)
and, end to end, against the sampler's own per-object layers."""
import ctypes
import functools

import numpy as np
import pytest

from oracle import stn_ref_c
from oracle import synth_pixel_ref as P
from oracle import synth_ref as S

CASES = {  # seed, first, B, canvas, counts, size range, gap, margin, share_size, sprites
    "mnist50": (1, 0, 120, 50, (1, 2, 3), (17, 23), 0, 0, False, 64),       # default Multi-MNIST of configs C2 / C4
    "crowded50": (2, 300, 60, 50, (3,), (30, 40), 0, 0, False, 64),        # restarts; sprites larger than their source
    "shared64": (3, 17, 80, 64, (1, 2, 3), (20, 25), 0, 0, True, 48),
    "gap1_margin2": (4, 0, 80, 50, (1, 2, 3), (17, 23), 1, 2, False, 64),
}
SPRITE_SIDE = 28


def sprites_for(c):
    from mog_asr_b200.dataset import default_sprites
    return default_sprites(c[9], SPRITE_SIDE, seed=9)


@functools.lru_cache(maxsize=None)
def oracle(name, max_restarts=32):
    seed, first, B, cs, counts, (smin, smax), gap, margin, share, _ = c = CASES[name]
    return P.place_pixels(sprites_for(c), seed, first, B, cs, list(counts), smin, smax, gap, margin, share, max_restarts=max_restarts)


def layers(sprites, cs, pos, size, sprite):
    """per-object masks [B, G, cs, cs] of what ``S.paste`` sums (before the live mask)"""
    B, G = sprite.shape
    U = np.asarray(sprites, np.float32)[sprite.reshape(-1)][..., None]
    v = stn_ref_c.forward(U, S.box_theta(pos, size, cs).reshape(B * G, 6), (cs, cs)).reshape(B, G, cs, cs)
    return np.clip(v, 0.0, 1.0) >= 0.05


def boxes_intersect(a, b):
    (x, y, w), (qx, qy, qw) = a, b
    return x < qx + qw and qx < x + w and y < qy + qw and qy < y + w


@pytest.mark.parametrize("name", sorted(CASES))
def test_oracle_placement_obeys_the_pixel_overlap_rule(name):
    seed, first, B, cs, counts, (smin, smax), gap, margin, share, nsp = c = CASES[name]
    num, pos, size, sprite = oracle(name)
    drawn = np.array([counts[S.draw_int(S.draw32(seed, first + b, 0, 0, 0, 7), 0, len(counts))] for b in range(B)])
    assert np.all(num <= drawn) and np.mean(num == drawn) > 0.9     # short only when every restart failed
    masks = layers(sprites_for(c), cs, pos, size, sprite)
    intersecting = 0
    for b in range(B):
        boxes = [(pos[b, g, 0], pos[b, g, 1], size[b, g, 0]) for g in range(num[b])]
        for (x, y, w) in boxes:
            assert smin <= w <= smax and margin <= x <= cs - w - margin and margin <= y <= cs - w - margin   # :171-172
        if share and boxes:
            assert len({w for _, _, w in boxes}) == 1
        assert np.all(sprite[b, :num[b]] < nsp) and np.all(pos[b, num[b]:] == 0) and np.all(size[b, num[b]:] == 0)
        for g in range(num[b]):
            assert masks[b, g].any()
            near = P.dilate(masks[b, g], gap)
            for k in range(g):
                assert not (near & masks[b, k]).any(), (b, g, k)
        intersecting += any(boxes_intersect(boxes[g], boxes[k]) for g in range(len(boxes)) for k in range(g))
    if name == "crowded50":
        # boxes overlap where pixels do not: the rule is not box intersection (mode "disjoint") in disguise
        assert intersecting > B // 4
        # and the case does exercise canvas restarts
        n1 = oracle(name, max_restarts=1)[0]
        assert np.sum(n1 < drawn) > B // 4
    # a canvas is a function of (seed, canvas index) only
    n2, p2, s2, sp2 = P.place_pixels(sprites_for(c), seed, first + 7, 10, cs, list(counts), smin, smax, gap, margin, share)
    assert np.array_equal(n2, num[7:17]) and np.array_equal(p2, pos[7:17]) and np.array_equal(s2, size[7:17])
    assert np.array_equal(sp2, sprite[7:17])


@pytest.fixture(scope="module")
def lib():
    from mog_asr_b200 import _lib, build
    build.build()
    return _lib.load()


def test_place_pixels_checks_arguments_before_any_launch(lib):
    from mog_asr_b200 import _lib
    one = 0x1000  # never dereferenced: validation fails first
    counts = (ctypes.c_int * 2)(1, 3)

    def call(B=4, canvas=50, max_objects=3, num_counts=2, size_min=17, size_max=23, gap=0, margin=0, sprites=one, side=28,
             num=one):
        return lib.mog_synth_place_pixels(1, 0, B, canvas, max_objects, counts, num_counts, size_min, size_max, gap, margin, 0,
                                          sprites, 8, side, one, one, num, one, one, one, None)

    assert call(canvas=0) == -2                                    # MOG_ERR_DIM
    assert call(size_max=16) == -2
    assert call(gap=-1) == -2
    assert call(side=0) == -2
    assert call(max_objects=2) == -2 and "exceeds max_objects" in _lib.last_error()
    assert call(canvas=129, size_max=23) == -4                     # MOG_ERR_UNSUPPORTED: > MOG_SYNTH_PIXEL_MAX_CANVAS
    assert "128" in _lib.last_error()
    assert call(sprites=None) == -1                                # MOG_ERR_NULL
    assert call(num=None) == -1
    # B = 0 is a no-op, whatever the pointers
    assert lib.mog_synth_place_pixels(1, 0, 0, 50, 3, counts, 2, 17, 23, 0, 0, 0, None, 8, 28, None, None, None, None, None, None,
                                      None) == 0


# ---- GPU ----------------------------------------------------------------------------------------------------------------
def device_dataset(name, device, mode="pixel"):
    from mog_asr_b200.dataset import DeviceMultiObjectDataset
    seed, first, B, cs, counts, srange, gap, margin, share, _ = c = CASES[name]
    return DeviceMultiObjectDataset(sprites_for(c), cs, counts, srange, gap, margin, mode, share, seed, device=device)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_cuda_pixel_placement_and_paste_match_oracle(name, cuda_device):
    seed, first, B, cs, counts, srange, gap, margin, share, _ = c = CASES[name]
    ds = device_dataset(name, cuda_device)
    num, pos, size, sprite = ds.place(first, B)
    rn, rp, rs, rsp = oracle(name)
    for got, want in ((num, rn), (pos, rp), (size, rs), (sprite, rsp)):
        assert np.array_equal(got.cpu().numpy(), want)
    img = ds.paste(num, pos, size, sprite).cpu().numpy()
    assert np.array_equal(img, S.paste(sprites_for(c), cs, rn, rp, rs, rsp))


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_cuda_pixel_placement_layers_through_the_sampler_never_touch(name, cuda_device):
    """end to end: the kernel's occupancy test equals what the sampler writes, so the device layers obey the rule"""
    import torch
    import torch.nn.functional as F
    from mog_asr_b200.transformer import transformer
    seed, first, B, cs, counts, srange, gap, margin, share, _ = CASES[name]
    ds = device_dataset(name, cuda_device)
    num, pos, size, sprite = ds.place(first, B)
    G = ds.G
    U = ds.sprites.index_select(0, sprite.reshape(-1).long()).unsqueeze(-1)
    v = transformer(U, ds.box_theta(pos, size, cs).reshape(B * G, 6), (cs, cs)).reshape(B, G, cs, cs)
    live = (torch.arange(G, device=cuda_device)[None, :] < num[:, None])[:, :, None, None]
    m = (torch.clamp(v, 0.0, 1.0) >= 0.05) & live
    assert int(m.sum(1).max()) <= 1                                             # no pixel in two layers
    assert bool((m.flatten(2).any(2) == live[:, :, 0, 0]).all())                # every live object left pixels
    if gap > 0:
        near = F.max_pool2d(m.float().reshape(B * G, 1, cs, cs), 2 * gap + 1, 1, gap).reshape(B, G, cs, cs) > 0
        others = m.sum(1, keepdim=True) - m.int() > 0
        assert not bool((near & others).any())                                   # nor within `gap` of another object


@pytest.mark.gpu
def test_cuda_pixel_placement_with_one_object_equals_disjoint(cuda_device):
    """the draws are shared and a lone object has nothing to clash with"""
    from mog_asr_b200.dataset import DeviceMultiObjectDataset, default_sprites
    sp = default_sprites(64, SPRITE_SIDE, seed=3)
    got = [DeviceMultiObjectDataset(sp, 64, (1,), (20, 25), 1, 2, mode, False, 21, device=cuda_device).place(1000, 3000)
           for mode in ("pixel", "disjoint")]
    for a, b in zip(*got):
        assert np.array_equal(a.cpu().numpy(), b.cpu().numpy())


@pytest.mark.gpu
def test_cuda_pixel_batches_split_over_ranks_and_grid_passes(cuda_device):
    import torch
    from mog_asr_b200.dataset import DeviceMultiObjectDataset
    ds = device_dataset("mnist50", cuda_device)
    # the launch caps the grid at 8 CTAs of 4 warps (one canvas each) per SM: this batch takes more than one grid pass
    per_pass = 32 * torch.cuda.get_device_properties(cuda_device).multi_processor_count
    B = 2 * ((per_pass + 200) // 2)
    assert B > per_pass
    whole = ds.batch(0, B)
    halves = [ds.batch(0, B // 2, rank=r, world=2) for r in range(2)]
    for k in ("images", "num", "pos", "size", "sprite"):
        assert torch.equal(torch.cat([h[k] for h in halves]), whole[k]), k
    # canvases of the second grid pass against the oracle
    seed, _, _, cs, counts, (smin, smax), gap, margin, share, _ = c = CASES["mnist50"]
    rn, rp, rs, rsp = P.place_pixels(sprites_for(c), seed, B - 40, 40, cs, list(counts), smin, smax, gap, margin, share)
    for k, want in (("num", rn), ("pos", rp), ("size", rs), ("sprite", rsp)):
        assert np.array_equal(whole[k][B - 40:].cpu().numpy(), want), k
    with pytest.raises(ValueError, match="canvas_size <= 128"):
        DeviceMultiObjectDataset(sprites_for(c), 130, (1,), (17, 23), mode="pixel", device=cuda_device)
