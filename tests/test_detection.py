"""Detection metrics (SURVEY §8(f) rank 4).  Parity here is PINNED: the golden vectors were produced by running the
reference's own ``evaluation_detection.evaluation`` (``tests/golden/make_golden_detection.py``)."""
import os

import numpy as np
import pytest

from oracle import detection_ref

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = ["detection_mnist", "detection_sprites", "detection_edge"]


def load(name):
    z = np.load(os.path.join(HERE, "golden", name + ".npz"))
    n = len(z["gt_num"])
    pos = [z["gt_pos"][k, :z["gt_num"][k]].reshape(-1).tolist() for k in range(n)]
    size = [z["gt_size"][k, :z["gt_num"][k]].reshape(-1).tolist() for k in range(n)]
    return z, pos, size


def random_case(seed, n, csize, max_gt, max_inf):
    rng = np.random.default_rng(seed)
    gt_num, inf_num = rng.integers(0, max_gt + 1, n), rng.integers(0, max_inf + 1, n)
    pos, size = [], []
    for k in range(n):
        wh = rng.integers(4, csize // 2, (gt_num[k], 2))
        xy = (rng.random((gt_num[k], 2)) * (csize - wh)).astype(np.int64)
        pos.append(xy.reshape(-1).tolist()); size.append(wh.reshape(-1).tolist())
    shifts = np.tanh(rng.normal(0, 0.5, (n, max_inf, 2))).astype(np.float32)
    scales = (1 / (1 + np.exp(-rng.normal(-0.5, 0.7, (n, max_inf, 1))))).astype(np.float32)
    return pos, size, shifts, scales, inf_num


@pytest.mark.parametrize("name", GOLDEN)
def test_oracle_matches_reference_golden(name):
    z, pos, size = load(name)
    got = detection_ref.evaluation(pos, size, z["inf_shifts"], z["inf_scales"], z["inf_num"], csize=int(z["csize"]))
    for g, key in zip(got, ("precision", "recall", "gt_max_iou", "detected_max_iou", "global_iou_mean")):
        assert np.array_equal(np.asarray(g), z[key]), key      # same float64 operations in the same order: bit-exact


@pytest.mark.gpu
@pytest.mark.parametrize("name", GOLDEN)
def test_cuda_matches_reference_golden(name, cuda_device):
    from mog_asr_b200 import detection
    z, pos, size = load(name)
    got = detection.evaluation(pos, size, z["inf_shifts"], z["inf_scales"], z["inf_num"], csize=int(z["csize"]), device=cuda_device)
    for g, key in zip(got[:4], ("precision", "recall", "gt_max_iou", "detected_max_iou")):
        assert np.array_equal(np.asarray(g), z[key]), key
    assert abs(got[4] - z["global_iou_mean"]) <= 1e-14        # matching found by DP, not scipy: equal optimum, ulp-level sum


@pytest.mark.gpu
@pytest.mark.parametrize("seed,n,csize,max_gt,max_inf", [(0, 512, 50, 3, 3), (1, 256, 64, 8, 8), (2, 300, 50, 8, 2), (3, 300, 50, 2, 8),
                                                           (4, 1, 50, 1, 1), (5, 64, 256, 6, 6)])
def test_cuda_per_instance_vs_oracle(seed, n, csize, max_gt, max_inf, cuda_device):
    import torch
    from mog_asr_b200 import detection
    pos, size, shifts, scales, inf_num = random_case(seed, n, csize, max_gt, max_inf)
    want = detection_ref.evaluation_per_instance(pos, size, shifts, scales, inf_num, csize=csize)
    P, S, num = detection.pack_ground_truth(pos, size)
    dev = torch.device(cuda_device)
    got = detection.detection_metrics(torch.tensor(P).to(dev), torch.tensor(S).to(dev), torch.tensor(num).to(dev), torch.tensor(shifts).to(dev),
                                      torch.tensor(scales).to(dev), torch.tensor(inf_num).to(dev), csize)
    got = [g.cpu().numpy() for g in got]
    for i in range(4):
        assert np.array_equal(got[i], want[i]), i
    np.testing.assert_allclose(got[4], want[4], rtol=0, atol=1e-14)


@pytest.mark.gpu
def test_cuda_rejects_too_many_boxes(cuda_device):
    import torch
    from mog_asr_b200 import detection
    dev = torch.device(cuda_device)
    z = lambda *s: torch.zeros(*s, device=dev)
    with pytest.raises(ValueError):
        detection.detection_metrics(z(2, 9, 2), z(2, 9, 2), z(2), z(2, 3, 2), z(2, 3), z(2), 50)


@pytest.mark.gpu
def test_non_integral_ground_truth_is_refused(cuda_device):
    """float ground-truth boxes with fractional coordinates would be truncated by the int32 kernel interface: refused."""
    import torch
    from mog_asr_b200 import detection
    pos = torch.tensor([[[3.5, 4.0]]], device=cuda_device)
    size = torch.tensor([[[10.0, 10.0]]], device=cuda_device)
    num = torch.tensor([1], device=cuda_device)
    sh = torch.zeros((1, 1, 2), device=cuda_device, dtype=torch.float64)
    sc = torch.full((1, 1), 0.3, device=cuda_device, dtype=torch.float64)
    with pytest.raises(ValueError):
        detection.detection_metrics(pos, size, num, sh, sc, num, 50)
    detection.detection_metrics(torch.floor(pos), size, num, sh, sc, num, 50)    # integral floats are fine


# ---------------------------------------------------------------------------------------------------------------------
# edges random boxes never reach: IoUs exactly on a threshold, ties in the matching, every (#gt, #inferred) pair and
# counts outside [0, G] / [0, T]; mog_detection_eval is called directly, its outputs NaN-filled first
# ---------------------------------------------------------------------------------------------------------------------
THRESHOLDS = [i * 0.05 + 0.5 for i in range(11)]          # :79, the reference's double arithmetic
CSIZE = 64                                                 # csize / 2 = 32: dyadic shifts and scales give exact boxes
# (w, h, mx, my, half, IoU as a fraction): ground truth (20, 20, w, h), inferred square centred on (mx, my) with half-side
# `half`, i.e. shift (m / 32 - 1), scale half / 32.  Found by an exhaustive CPU search over w, h <= 20, centres 14 ... 38 and
# half-sides 0.5 ... 11: every threshold but i = 7 is hit; that one is 0.8500000000000001, above the double nearest 0.85,
# and no small box pair rounds to it.  17/20 rounds to the double nearest 0.85, so it counts at 0.8 and not at i = 7.
PLANTED = [(2, 2, 20, 21, 1.0, (1, 2)), (5, 9, 21, 24, 3.5, (11, 20)), (2, 3, 21, 21, 1.5, (3, 5)), (12, 19, 26, 26, 6.0, (13, 20)),
           (6, 9, 23, 23, 3.0, (7, 10)), (2, 3, 21, 21, 1.0, (3, 4)), (3, 4, 21, 22, 2.0, (4, 5)), (16, 19, 28, 28, 8.0, (17, 20)),
           (8, 9, 24, 24, 4.0, (9, 10)), (18, 19, 29, 29, 9.0, (19, 20)), (2, 2, 21, 21, 1.0, (1, 1)), (6, 6, 23, 23, 3.0, (1, 1))]


def planted_box(w, h, mx, my, half):
    """ground-truth position and size, and the inferred (shift x, shift y, scale)"""
    return (20, 20), (w, h), (mx / (CSIZE / 2) - 1, my / (CSIZE / 2) - 1, half / (CSIZE / 2))


def oracle_iou(pos, size, shift_scale):
    """the IoU of one pair through the oracle's own box arithmetic"""
    cx, cy, s = shift_scale
    return detection_ref.evaluation_per_instance([list(pos)], [list(size)], [[[cx, cy]]], [[[s]]], [1], csize=CSIZE)[2][0]


def test_planted_ious_sit_on_their_thresholds():
    """Each planted IoU is the double of its fraction, and the fractions hit thresholds 0.5, 0.55, 0.6, 0.65, 0.7, 0.75,
    0.8, 0.9, 0.95 and 1.0 bit for bit (gt_max_iou of a one-pair image is that pair's IoU).  Strict >: a pair on threshold
    i counts at every threshold below i and at none from i on; a perfect detection does not count at 1.0."""
    hit = set()
    for w, h, mx, my, half, (p, q) in PLANTED:
        pos, size, ss = planted_box(w, h, mx, my, half)
        iou = oracle_iou(pos, size, ss)
        assert iou == p / q, (w, h, mx, my, half)
        prec = detection_ref.evaluation_per_instance([list(pos)], [list(size)], [[ss[:2]]], [[[ss[2]]]], [1], csize=CSIZE)[0][0]
        assert np.array_equal(prec, (iou > np.array(THRESHOLDS)).astype(float))
        hit |= {i for i, t in enumerate(THRESHOLDS) if iou == t}
    assert hit == set(range(11)) - {7}
    assert 17 / 20 < THRESHOLDS[7] and 17 / 20 > THRESHOLDS[6]


def det_eval(pos, size, gt_num, shifts, scales, inf_num, dev):
    """mog_detection_eval on [B][G][2] int boxes, [B][T][2] shifts, [B][T] scales, with NaN-filled outputs"""
    import torch
    from mog_asr_b200 import _lib
    B, G, T = pos.shape[0], pos.shape[1], shifts.shape[1]
    t = [torch.tensor(np.ascontiguousarray(a), device=dev) for a in (pos.astype(np.int32), size.astype(np.int32), np.asarray(gt_num, np.int32),
                                                                      shifts.astype(np.float64), scales.astype(np.float64),
                                                                      np.asarray(inf_num, np.int32))]
    out = [torch.full(s, float("nan"), dtype=torch.float64, device=dev) for s in ((B, 11), (B, 11), (B,), (B,), (B,))]
    rc = _lib.load().mog_detection_eval(*(a.data_ptr() for a in t), B, G, T, float(CSIZE), *(o.data_ptr() for o in out),
                                        torch.cuda.current_stream(dev).cuda_stream)
    torch.cuda.synchronize(dev)
    assert rc == 0, _lib.last_error()
    return [o.cpu().numpy() for o in out]


def assert_matches_oracle(got, pos, size, gt_num, shifts, scales, inf_num):
    """precision, recall and both max-IoU means bit for bit, the matched IoU to 1e-14; counts clamped as the header says"""
    G, T = pos.shape[1], shifts.shape[1]
    ng, ni = np.clip(gt_num, 0, G), np.clip(inf_num, 0, T)
    want = detection_ref.evaluation_per_instance([pos[k, :ng[k]].reshape(-1).tolist() for k in range(len(ng))],
                                                 [size[k, :ng[k]].reshape(-1).tolist() for k in range(len(ng))],
                                                 shifts, scales[..., None], ni, csize=CSIZE)
    for i in range(4):
        assert np.array_equal(got[i], want[i]), i
    np.testing.assert_allclose(got[4], want[4], rtol=0, atol=1e-14)


@pytest.mark.gpu
def test_cuda_exact_thresholds(cuda_device):
    """One planted pair per image, and the same pairs two or three to an image; the kernel must agree with the oracle on
    which side of each threshold they fall, perfect detections at 1.0 and 17/20 at 0.8500000000000001 included."""
    n = len(PLANTED)
    pos, size = np.zeros((n + 4, 3, 2), np.int64), np.zeros((n + 4, 3, 2), np.int64)
    shifts, scales = np.full((n + 4, 3, 2), np.nan), np.full((n + 4, 3), np.nan)
    gt_num, inf_num = np.zeros(n + 4, np.int64), np.zeros(n + 4, np.int64)
    for k, case in enumerate(PLANTED):
        p, s, ss = planted_box(*case[:5])
        pos[k, 0], size[k, 0], shifts[k, 0], scales[k, 0] = p, s, ss[:2], ss[2]
        gt_num[k] = inf_num[k] = 1
    for k in range(4):                                      # several planted pairs, moved apart by whole pixels (exact)
        for j in range(2 + k % 2):
            w, h, mx, my, half, _ = PLANTED[(3 * k + 5 * j) % n]
            dx, dy = 12 * j - 8, 10 * j - 6
            p, s, ss = planted_box(w, h, mx + dx, my + dy, half)
            pos[n + k, j], size[n + k, j], shifts[n + k, j], scales[n + k, j] = (p[0] + dx, p[1] + dy), s, ss[:2], ss[2]
        gt_num[n + k] = inf_num[n + k] = 2 + k % 2
    got = det_eval(pos, size, gt_num, shifts, scales, inf_num, cuda_device)
    assert_matches_oracle(got, pos, size, gt_num, shifts, scales, inf_num)
    for k, (*_, (p, q)) in enumerate(PLANTED):
        assert got[2][k] == p / q
        assert np.array_equal(got[0][k], (p / q > np.array(THRESHOLDS)).astype(float)), k
    perfect = [k for k, c in enumerate(PLANTED) if c[5] == (1, 1)]
    assert perfect and np.all(got[0][perfect, 10] == 0) and np.all(got[0][perfect, 9] == 1)
    assert [got[0][k, 6:8].tolist() for k, c in enumerate(PLANTED) if c[5] == (17, 20)] == [[1.0, 0.0]]


@pytest.mark.gpu
def test_cuda_matching_ties(cuda_device):
    """Duplicate inferred boxes, duplicate ground truths, one detection overlapping two ground truths equally (mirror
    images about its centre), and eight identical boxes on each side (every pair tied, the eight-term sums)."""
    c = lambda m: m / (CSIZE / 2) - 1
    images = [
        ([(20, 20, 10, 12), (26, 18, 9, 9)], [(c(26), c(26), 6 / 32)] * 3),                  # three identical detections
        ([(20, 24, 8, 10), (36, 24, 8, 10)], [(c(32), c(29), 6 / 32)]),                        # one detection, two equal IoUs
        ([(20, 24, 8, 10), (36, 24, 8, 10)], [(c(32), c(29), 6 / 32), (c(32), c(29), 6 / 32)]),
        ([(18, 18, 12, 12)] * 3, [(c(24), c(24), 6 / 32), (c(25), c(24), 6 / 32), (c(24), c(24), 6 / 32)]),
        ([(18, 18, 12, 12)] * 8, [(c(25), c(23), 5.5 / 32)] * 8),
        ([(18, 18, 12, 12)] * 8, [(c(25), c(23), 5.5 / 32)] * 5),
        ([(18, 18, 12, 12)] * 5, [(c(25), c(23), 5.5 / 32)] * 8),
        ([(10, 10, 6, 6), (30, 30, 6, 6), (10, 10, 6, 6)], [(c(13), c(13), 3 / 32), (c(33), c(33), 3 / 32), (c(14), c(13), 3 / 32),
                                                             (c(33), c(33), 3 / 32)]),
    ]
    B = len(images)
    pos, size = np.zeros((B, 8, 2), np.int64), np.zeros((B, 8, 2), np.int64)
    shifts, scales = np.full((B, 8, 2), np.nan), np.full((B, 8), np.nan)
    gt_num, inf_num = np.zeros(B, np.int64), np.zeros(B, np.int64)
    for k, (gts, dets) in enumerate(images):
        for j, (x, y, w, h) in enumerate(gts):
            pos[k, j], size[k, j] = (x, y), (w, h)
        for j, (cx, cy, s) in enumerate(dets):
            shifts[k, j], scales[k, j] = (cx, cy), s
        gt_num[k], inf_num[k] = len(gts), len(dets)
    got = det_eval(pos, size, gt_num, shifts, scales, inf_num, cuda_device)
    assert_matches_oracle(got, pos, size, gt_num, shifts, scales, inf_num)
    det = images[1][1][0]
    assert oracle_iou((20, 24), (8, 10), det) == oracle_iou((36, 24), (8, 10), det) > 0


def random_boxes(rng, B, G, T):
    """random integer ground truth and float64-widened fp32 inferred boxes at csize 64, every slot filled"""
    wh = rng.integers(2, CSIZE // 2, (B, G, 2))
    xy = (rng.random((B, G, 2)) * (CSIZE - wh)).astype(np.int64)
    shifts = np.tanh(rng.normal(0, 0.5, (B, T, 2))).astype(np.float32).astype(np.float64)
    scales = (1 / (1 + np.exp(-rng.normal(-0.5, 0.7, (B, T))))).astype(np.float32).astype(np.float64)
    return xy, wh, shifts, scales


@pytest.mark.gpu
def test_cuda_every_box_count_pair(cuda_device):
    """All 81 (#gt, #inferred) pairs in 0..8 x 0..8 with G = T = 8, three images each, in one launch of four 64-thread
    CTAs.  Slots past an image's counts hold boxes too (inferred ones NaN): they must not be read."""
    rng = np.random.default_rng(81)
    pairs = [(r, c) for r in range(9) for c in range(9)] * 3
    B = len(pairs)
    pos, size, shifts, scales = random_boxes(rng, B, 8, 8)
    gt_num, inf_num = np.array([p[0] for p in pairs]), np.array([p[1] for p in pairs])
    for k in range(B):
        shifts[k, inf_num[k]:], scales[k, inf_num[k]:] = np.nan, np.nan
    assert B > 3 * 64
    got = det_eval(pos, size, gt_num, shifts, scales, inf_num, cuda_device)
    assert_matches_oracle(got, pos, size, gt_num, shifts, scales, inf_num)


@pytest.mark.gpu
def test_cuda_counts_outside_the_range_are_clamped(cuda_device):
    """gt_num of G + 3 and -1, inf_num of T + 2 and -1 give the bits of the clamped counts (the header clamps them to
    [0, G] / [0, T]; nothing past the padded arrays is read)."""
    rng = np.random.default_rng(5)
    B, G, T = 96, 5, 4
    pos, size, shifts, scales = random_boxes(rng, B, G, T)
    gt_num, inf_num = rng.integers(0, G + 1, B), rng.integers(0, T + 1, B)
    gt_num[0::4], gt_num[1::4] = G + 3, -1
    inf_num[2::4], inf_num[0::8] = T + 2, -1
    got = det_eval(pos, size, gt_num, shifts, scales, inf_num, cuda_device)
    clamped = det_eval(pos, size, np.clip(gt_num, 0, G), shifts, scales, np.clip(inf_num, 0, T), cuda_device)
    for a, b in zip(got, clamped):
        assert np.array_equal(a.view(np.uint64), b.view(np.uint64))
    assert_matches_oracle(got, pos, size, gt_num, shifts, scales, inf_num)
