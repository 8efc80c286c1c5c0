"""Synthetic-dataset feeder, rotated objects with tight-box labels (``DeviceMultiObjectDataset(..., angles=...)``,
``mog_synth_place_rotated``): the reference rotates each object and labels it with its re-cropped tight box
(multi_mnist.py:144-163).  Checked against oracle/synth_rotated_ref.place_rotated (same counter-based draws, candidates
evaluated on the full canvas with the C sampler oracle) in every rule, and, with the single angle 0, against the
unrotated pixel-overlap placement."""
import ctypes
import functools

import numpy as np
import pytest

from oracle import synth_pixel_ref as P
from oracle import synth_ref as S
from oracle import synth_rotated_ref as R

SPRITE_SIDE = 28
MODES = {"bbox": 0, "disjoint": 1, "pixel": 2}


def angle_set(name):
    from mog_asr_b200.dataset import dsprites_angles
    return {"pm30": tuple(float(a) for a in np.linspace(-30.0, 30.0, 61)), "dsprites": dsprites_angles(), "zero": (0.0,)}[name]


def rot_of(name):
    from mog_asr_b200.dataset import rotation_table
    return rotation_table(angle_set(name))


CASES = {  # seed, first, B, canvas, counts, size range, gap, margin, share_size, sprites, angles, blank sprites
    "mnist50": (1, 0, 80, 50, (1, 2, 3), (17, 23), 0, 0, False, 64, "pm30", False),     # configs C2 / C4
    "dsprites64": (6, 40, 60, 64, (1, 2, 3), (20, 25), 0, 0, False, 64, "dsprites", False),
    "crowded50": (2, 300, 40, 50, (3,), (24, 30), 0, 0, False, 64, "dsprites", False),   # restarts
    "shared64": (3, 17, 60, 64, (1, 2, 3), (20, 25), 0, 0, True, 48, "pm30", False),
    "gap1_margin2": (4, 0, 60, 50, (1, 2, 3), (17, 23), 1, 2, False, 64, "dsprites", False),
    "blank64": (5, 0, 60, 64, (2, 3), (20, 25), 1, 0, False, 16, "pm30", True),          # every third sprite is blank
}


def sprites_for(c):
    from mog_asr_b200.dataset import default_sprites
    sp = default_sprites(c[9], SPRITE_SIDE, seed=9)
    if c[11]:
        sp[::3] = 0.0
    return sp


@functools.lru_cache(maxsize=None)
def oracle(name, mode, max_restarts=32):
    seed, first, B, cs, counts, (smin, smax), gap, margin, share, _, ang, _ = c = CASES[name]
    return R.place_rotated(sprites_for(c), rot_of(ang), seed, first, B, cs, list(counts), smin, smax, gap, margin, MODES[mode],
                           share, max_restarts=max_restarts)


def check_placement(sprites, cs, counts, gap, margin, mode, seed, first, placement):
    """the properties every placement must have, from full-canvas forwards of the returned theta"""
    num, pos, size, sprite, theta, square = placement
    B = num.shape[0]
    drawn = np.array([counts[S.draw_int(S.draw32(seed, first + b, 0, 0, 0, 7), 0, len(counts))] for b in range(B)])
    assert np.all(num <= drawn)
    for b in range(B):
        n = num[b]
        assert np.all(pos[b, n:] == 0) and np.all(size[b, n:] == 0) and np.all(sprite[b, n:] == 0) and np.all(theta[b, n:] == 0)
        masks = [R.masks_of(sprites, sprite[b, g], theta[b, g], cs)[0] for g in range(n)]
        for g in range(n):
            x, y, w, h = pos[b, g, 0], pos[b, g, 1], size[b, g, 0], size[b, g, 1]
            sx, sy, e = square[b, g]
            assert margin <= x and x + w <= cs - margin and margin <= y and y + h <= cs - margin and w > 0 and h > 0
            m = masks[g]
            if m.any():
                assert R.tight_box(m) == (x, y, w, h)
                ys, xs = np.nonzero(m)
                assert xs.min() >= sx - 1 and xs.max() <= sx + e and ys.min() >= sy - 1 and ys.max() <= sy + e
            else:
                assert (x, y, w, h) == (sx, sy, e, e)
        for g in range(n):
            for k in range(g):
                if mode == "pixel":
                    assert not (P.dilate(masks[g], gap) & masks[k]).any(), (b, g, k)
                elif masks[g].any() and masks[k].any():
                    assert not S.boxes_clash(MODES[mode], *pos[b, g], *size[b, g], *pos[b, k], *size[b, k], gap), (b, g, k)
    return drawn


# ---- CPU: the oracle ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", sorted(MODES))
@pytest.mark.parametrize("canvas", [50, 64])
@pytest.mark.parametrize("angles", ["pm30", "dsprites"])
def test_oracle_rotated_placement_obeys_its_rule(angles, canvas, mode):
    from mog_asr_b200.dataset import default_sprites
    counts, srange = (1, 2, 3), ((17, 23) if canvas == 50 else (20, 25))
    sp = default_sprites(32, SPRITE_SIDE, seed=9)
    placement = R.place_rotated(sp, rot_of(angles), 11, 5, 30, canvas, list(counts), *srange, 0, 0, MODES[mode])
    drawn = check_placement(sp, canvas, counts, 0, 0, mode, 11, 5, placement)
    num, _, size, _, _, _ = placement
    assert np.mean(num == drawn) > 0.5
    live = np.arange(size.shape[1])[None, :] < num[:, None]
    assert np.any(size[live][:, 0] != size[live][:, 1])                 # tight boxes are not squares in general


@pytest.mark.parametrize("name", sorted(CASES))
def test_oracle_rotated_cases_obey_their_rules(name):
    seed, first, B, cs, counts, srange, gap, margin, share, _, _, blank = c = CASES[name]
    for mode in MODES:
        num, pos, size, sprite, theta, square = placement = oracle(name, mode)
        drawn = check_placement(sprites_for(c), cs, counts, gap, margin, mode, seed, first, placement)
        live = np.arange(sprite.shape[1])[None, :] < num[:, None]
        if blank:                                                        # blank objects are labelled with their e-square
            empty = live & (sprite % 3 == 0)
            assert empty.any() and np.array_equal(pos[empty], square[empty][:, :2])
            assert np.all(size[empty] == square[empty][:, 2:])
    if name == "crowded50":
        n1 = oracle(name, "pixel", max_restarts=1)[0]
        assert np.sum(n1 < drawn) > B // 4                               # the case exercises canvas restarts


@pytest.mark.parametrize("canvas", [50, 64])
def test_theta_at_angle_zero_is_box_theta_bit_for_bit(canvas):
    ws = np.arange(2, 31)
    ps = np.arange(0, canvas - 1)
    for w in ws:
        got = np.stack([R.rotated_theta(1.0, 0.0, int(w), int(w), int(x), int(y), canvas) for x in ps for y in ps[::7]])
        xy = np.array([(x, y) for x in ps for y in ps[::7]], np.int32)
        want = S.box_theta(xy, np.full_like(xy, w), canvas)
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), w          # signed zeros included
    assert R.extent(23, 1.0, 0.0, canvas) == 23


def test_oracle_at_angle_zero_is_the_pixel_placement_with_tight_boxes():
    seed, first, B, cs, counts, (smin, smax), gap, margin, share, _, _, _ = c = CASES["gap1_margin2"]
    sp = sprites_for(c)
    num, pos, size, sprite, theta, square = R.place_rotated(sp, rot_of("zero"), seed, first, B, cs, list(counts), smin, smax, gap,
                                                            margin, 2, share)
    rn, rp, rs, rsp = P.place_pixels(sp, seed, first, B, cs, list(counts), smin, smax, gap, margin, share)
    assert np.array_equal(num, rn) and np.array_equal(sprite, rsp)
    live = np.arange(rp.shape[1])[None, :] < rn[:, None]
    assert np.array_equal(square[live][:, :2], rp[live]) and np.array_equal(square[live][:, 2], rs[live][:, 0])
    want = S.box_theta(rp, rs, cs)
    assert np.array_equal(theta[live].view(np.uint32), want[live].view(np.uint32))
    assert np.all(pos[live] >= rp[live]) and np.all(pos[live] + size[live] <= rp[live] + rs[live])   # inside the old square


def test_angle_tables():
    from mog_asr_b200.dataset import dsprites_angles, rotation_table
    a = dsprites_angles()
    assert len(a) == 40 and a[0] == 0.0 and a[-1] == 360.0
    t = rotation_table((0.0, 90.0))
    assert t.dtype == np.float64 and t[0, 0] == 1.0 and t[0, 1] == 0.0 and not np.signbit(t[0, 1])
    assert abs(t[1, 0]) < 1e-15 and t[1, 1] == 1.0


@pytest.fixture(scope="module")
def lib():
    from mog_asr_b200 import _lib, build
    build.build()
    return _lib.load()


def test_place_rotated_checks_arguments_before_any_launch(lib):
    from mog_asr_b200 import _lib
    one = 0x1000  # never dereferenced: validation fails first
    counts = (ctypes.c_int * 2)(1, 3)
    unit = (ctypes.c_double * 4)(1.0, 0.0, 0.0, 1.0)

    def call(B=4, canvas=50, max_objects=3, size_min=17, size_max=23, gap=0, mode=2, sprites=one, side=28, rot=unit, A=2,
             num=one, theta=one):
        return lib.mog_synth_place_rotated(1, 0, B, canvas, max_objects, counts, 2, size_min, size_max, gap, 0, mode, 0,
                                           sprites, 8, side, rot, A, num, one, one, one, theta, None)

    assert call(canvas=0) == -2                                    # MOG_ERR_DIM
    assert call(canvas=1, size_max=17) == -2
    assert call(size_min=1) == -2                                  # a size-1 object has no finite theta
    assert call(size_max=16) == -2
    assert call(gap=-1) == -2
    assert call(side=0) == -2
    assert call(mode=3) == -2 and call(mode=-1) == -2
    assert call(A=0) == -2 and call(A=65) == -2
    assert call(max_objects=2) == -2 and "exceeds max_objects" in _lib.last_error()
    bad = (ctypes.c_double * 4)(1.0, 0.0, 0.6, 0.6)
    assert call(rot=bad) == -2 and "unit" in _lib.last_error()
    nan = (ctypes.c_double * 2)(float("nan"), 0.0)
    assert call(rot=nan, A=1) == -2
    assert call(canvas=129) == -4                                  # MOG_ERR_UNSUPPORTED: > MOG_SYNTH_PIXEL_MAX_CANVAS
    assert "128" in _lib.last_error()
    for kw in ("sprites", "rot", "num", "theta"):
        assert call(**{kw: None}) == -1                            # MOG_ERR_NULL
    # B = 0 is a no-op, whatever the pointers
    assert lib.mog_synth_place_rotated(1, 0, 0, 50, 3, counts, 2, 17, 23, 0, 0, 2, 0, None, 8, 28, None, 2, None, None, None,
                                       None, None, None) == 0


# ---- GPU ----------------------------------------------------------------------------------------------------------------
def device_dataset(name, device, mode, angles="case"):
    """``angles``: "case" for the case's set, else what the dataset takes (None: unrotated)"""
    from mog_asr_b200.dataset import DeviceMultiObjectDataset
    seed, first, B, cs, counts, srange, gap, margin, share, _, ang, _ = c = CASES[name]
    return DeviceMultiObjectDataset(sprites_for(c), cs, counts, srange, gap, margin, mode, share, seed, device=device,
                                    angles=angle_set(ang) if angles == "case" else angles)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", sorted(MODES))
@pytest.mark.parametrize("name", sorted(CASES))
def test_cuda_rotated_placement_and_paste_match_oracle(name, mode, cuda_device):
    seed, first, B, cs, counts, srange, gap, margin, share, _, _, _ = c = CASES[name]
    ds = device_dataset(name, cuda_device, mode)
    num, pos, size, sprite, theta = ds.place(first, B)
    rn, rp, rs, rsp, rth, _ = oracle(name, mode)
    for k, got, want in (("num", num, rn), ("pos", pos, rp), ("size", size, rs), ("sprite", sprite, rsp)):
        assert np.array_equal(got.cpu().numpy(), want), k
    assert np.array_equal(theta.cpu().numpy().view(np.uint32), rth.view(np.uint32))
    img = ds.paste(num, pos, size, sprite, theta).cpu().numpy()
    assert np.array_equal(img, R.paste(sprites_for(c), cs, rn, rsp, rth))


@pytest.mark.gpu
@pytest.mark.parametrize("mode", sorted(MODES))
def test_cuda_rotated_batches_split_over_ranks_and_grid_passes(mode, cuda_device):
    import torch
    ds = device_dataset("mnist50", cuda_device, mode)
    # the launch caps the grid at 8 CTAs of 4 warps (one canvas each) per SM: this batch takes more than one grid pass
    per_pass = 32 * torch.cuda.get_device_properties(cuda_device).multi_processor_count
    B = 2 * ((per_pass + 200) // 2)
    assert B > per_pass
    whole = ds.batch(0, B)
    halves = [ds.batch(0, B // 2, rank=r, world=2) for r in range(2)]
    for k in ("images", "num", "pos", "size", "sprite", "theta"):
        assert torch.equal(torch.cat([h[k] for h in halves]), whole[k]), k
    seed, _, _, cs, counts, (smin, smax), gap, margin, share, _, ang, _ = c = CASES["mnist50"]
    want = R.place_rotated(sprites_for(c), rot_of(ang), seed, B - 40, 40, cs, list(counts), smin, smax, gap, margin, MODES[mode],
                           share)
    for k, w in zip(("num", "pos", "size", "sprite", "theta"), want):
        assert np.array_equal(whole[k][B - 40:].cpu().numpy(), w), k


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["mnist50", "gap1_margin2", "shared64", "blank64"])
def test_cuda_angle_zero_reproduces_the_pixel_feeder(name, cuda_device):
    import torch
    B = 2000
    rot = device_dataset(name, cuda_device, "pixel", angles=(0.0,)).batch(0, B)
    old = device_dataset(name, cuda_device, "pixel", angles=None)
    assert old.angles is None
    ref = old.batch(0, B)
    for k in ("num", "sprite", "images"):
        assert torch.equal(rot[k], ref[k]), k
    live = (torch.arange(old.G, device=cuda_device)[None, :] < ref["num"][:, None])
    # against the fp64 expression on the host: the device box_theta (torch on the GPU) is not always correctly rounded;
    # it gives t12 = 2.9e-16 where the centre is exactly 0 (the canvases above agree all the same)
    want = S.box_theta(ref["pos"].cpu().numpy(), ref["size"].cpu().numpy(), old.cs)
    assert np.array_equal(rot["theta"].cpu().numpy()[live.cpu().numpy()].view(np.uint32), want[live.cpu().numpy()].view(np.uint32))
    assert bool((rot["pos"][live] >= ref["pos"][live]).all())
    assert bool((rot["pos"][live] + rot["size"][live] <= ref["pos"][live] + ref["size"][live]).all())


@pytest.mark.gpu
def test_cuda_dataset_rejects_bad_angle_sets(cuda_device):
    from mog_asr_b200.dataset import DeviceMultiObjectDataset
    sp = np.zeros((2, 8, 8), np.float32)
    for angles in ((), tuple(range(65))):
        with pytest.raises(ValueError, match="1 to 64"):
            DeviceMultiObjectDataset(sp, 50, (1,), (3, 5), device=cuda_device, angles=angles)
    with pytest.raises(ValueError, match="canvas_size <= 128"):
        DeviceMultiObjectDataset(sp, 130, (1,), (3, 5), mode="disjoint", device=cuda_device, angles=(0.0,))


@pytest.mark.gpu
def test_evaluate_detection_runs_on_a_rotated_batch(cuda_device):
    import torch
    from mog_asr_b200.air import AIRModel, CudaOps, config_from_flags, evaluate_detection
    from mog_asr_b200.dataset import DeviceMultiObjectDataset, default_sprites, dsprites_angles
    cfg = config_from_flags("mnist", "13")
    torch.manual_seed(0)
    model = AIRModel(cfg, ops=CudaOps()).to(cuda_device)
    ds = DeviceMultiObjectDataset(default_sprites(32, 28, seed=2), 50, (1, 2, 3), (11, 15), mode="pixel", seed=4,
                                  device=cuda_device, angles=dsprites_angles())
    batch = ds.batch(0, 96)
    assert bool((batch["size"][:, :, 0] != batch["size"][:, :, 1]).any())
    res = evaluate_detection(model, batch)
    for k in ("precision", "recall"):
        assert res[k].shape == (11,) and bool(torch.isfinite(res[k]).all())
    for k in ("gt_max_iou", "detected_max_iou", "global_iou"):
        assert 0.0 <= float(res[k]) <= 1.0
    assert 0.0 <= float(res["accuracy"]) <= 1.0
