"""GPU parity of the ASR regulariser kernels (csrc/mog_asr.cu: mog_asr_reg_colsum, mog_asr_reg_forward, mog_asr_reg_backward)
against oracle/asr_ref.py in fp64, at TF's sub-gradient ties, at the gates, step and count limits and batch sizes around the
128-thread block edge, past one grid pass of the column sum, in the data-parallel form, and at confident z_pres.

The C ABI is called directly, on the current stream.  Every output the header says is fully written (per_image, components,
margin and the three gradients) is pre-filled with NaN, so an element a kernel never writes fails the comparison.  psum is
always passed explicitly and the oracle gets ``batch_prob_mean = psum * inv_global_batch``, so the forward and backward are
checked apart from the column sum, which has a test of its own.

Bounds are per entry.  On inputs exact in fp32 (canvas 64, scales k/64, dyadic shifts, gammas and g_per_image, T a power of
two) the kernel and the oracle take the same branch at every tie, and the geometry values and gradients are bit-equal to the
oracle.  Elsewhere an entry is held to ``ULPS * 2^-23 * depth * sum|terms|``: the sum of the magnitudes of the operands that
enter it, times the number of roundings it accumulates through.  The terms that depend on P = sigmoid(log-odds) carry the
conditioning of the fp32 P: log(1 - P) turns the few-ulp error of P into an absolute error of P / (1 - P) ulp.  Above
|log-odds| of about 8 that is the whole story -- fp32 P differs from the fp64 one by more than the quantity measured, and from
about 16.6 up it is exactly 1 -- so confident z_pres is checked against the header's formulas evaluated in fp64 on the
fp32-rounded P instead of against the fp64 oracle."""
import ctypes

import numpy as np
import pytest
import torch

from mog_asr_b200 import _lib
from oracle import asr_ref
from tests import helpers as H

pytestmark = pytest.mark.gpu

EPS32 = H.EPS32
FLT_MIN = 2.0 ** -126
ULPS = 4
F32, F64 = np.float32, np.float64
COMPONENTS = ("pr_num", "num_min", "area", "out", "size", "overlap")
GAMMAS = ("gamma_num", "gamma_margin", "gamma_elem", "gamma_bbox", "gamma_size", "gamma_area")


# ---------------------------------------------------------------------------------------------------------------------
# calling the kernels
# ---------------------------------------------------------------------------------------------------------------------
def c_config(cfg):
    c = _lib.AsrConfig()
    c.canvas_size = cfg["canvas_size"]
    c.max_steps = cfg["max_steps"]
    c.num_counts = len(cfg["counts"])
    for i, v in enumerate(cfg["counts"]):
        c.counts[i] = v
    for k in GAMMAS:
        setattr(c, k, cfg.get(k, 0.0))
    c.size_min, c.size_max = cfg.get("area_minmax", (0.0, 0.0))
    return c


def call(fn, *args):
    rc = fn(*args, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert rc == 0, _lib.last_error()


def ptr(t):
    return t.data_ptr() if t is not None else None


def nan_buffer(shape, dev):
    return torch.full(shape, float("nan"), device=dev)


def to_dev(case, dev):
    return {k: torch.from_numpy(np.ascontiguousarray(case[k])).to(dev) for k in ("lo", "sh", "sc", "gp", "gm", "psum")}


def forward(L, d, case, cfg, components=True):
    B, T = case["lo"].shape
    dev = d["lo"].device
    per_image, margin = nan_buffer((B,), dev), nan_buffer((1,), dev)
    comps = nan_buffer((B, _lib.MOG_ASR_NUM_COMPONENTS), dev) if components else None
    call(L.mog_asr_reg_forward, ptr(d["lo"]), ptr(d["sh"]), ptr(d["sc"]), ptr(d["psum"]), float(case["inv_B"]), B, T,
         ctypes.byref(c_config(cfg)), ptr(per_image), ptr(comps), ptr(margin))
    return per_image, comps, margin


def backward(L, d, case, cfg, g_margin="given"):
    """g_margin: "given" passes case["gm"], "zero" a device 0.0, None a NULL pointer"""
    B, T = case["lo"].shape
    dev = d["lo"].device
    gm = {"given": d["gm"], "zero": torch.zeros(1, device=dev), None: None}[g_margin]
    d_lo, d_sh, d_sc = nan_buffer((B, T), dev), nan_buffer((B, T, 2), dev), nan_buffer((B, T), dev)
    call(L.mog_asr_reg_backward, ptr(d["lo"]), ptr(d["sh"]), ptr(d["sc"]), ptr(d["psum"]), float(case["inv_B"]), ptr(d["gp"]),
         ptr(gm), B, T, ctypes.byref(c_config(cfg)), ptr(d_lo), ptr(d_sh), ptr(d_sc))
    return d_lo, d_sh, d_sc


def np_(t):
    return t.detach().cpu().numpy()


# ---------------------------------------------------------------------------------------------------------------------
# references and bounds
# ---------------------------------------------------------------------------------------------------------------------
def pbar_of(case):
    return case["psum"].astype(F64) * F64(case["inv_B"])


def oracle(case, cfg):
    """asr_numpy with batch_prob_mean = psum * inv_global_batch.  The oracle takes that mean as a constant; the kernels
    differentiate it as the mean it stands for, psum[t] = sum_b P[b,t] over the global batch (:982), so the margin's
    gradient d margin / d pbar[t] * inv_global_batch * P (1 - P) is added to each image's d_log_odds."""
    T = case["lo"].shape[1]
    kw = {k: cfg[k] for k in GAMMAS if k in cfg}
    geo = dict(canvas_size=cfg["canvas_size"], counts=list(cfg["counts"]), max_steps=T, area_minmax=cfg.get("area_minmax", (0.0, 0.0)))
    r = asr_ref.asr_numpy(case["lo"], case["sh"], case["sc"], g_per_image=case["gp"], g_margin=float(case["gm"][0]),
                          batch_prob_mean=torch.tensor(pbar_of(case)), **geo, **kw)
    if cfg.get("gamma_margin", 0.0) > 1e-8:
        pb = torch.tensor(pbar_of(case), requires_grad=True)
        lo, sh, sc = (torch.tensor(case[k], dtype=torch.float64) for k in ("lo", "sh", "sc"))
        (dm,) = torch.autograd.grad(asr_ref.asr_terms(lo, sh, sc, batch_prob_mean=pb, **geo, **kw)["margin"], pb)
        P = r["P"]
        r["d_log_odds"] = r["d_log_odds"] + float(case["gm"][0]) * dm.numpy() * F64(case["inv_B"]) * P * (1 - P)
    return r


def sigmoid64(x):
    return 0.5 * (1.0 + np.tanh(0.5 * x))


def logit_eps(p):
    return np.log(p + 1e-8) - np.log(1.0 - p + 1e-8)


def dlogit_eps(p):
    return 1.0 / (p + 1e-8) + 1.0 / (1.0 - p + 1e-8)


def bce_logits(z, x):
    return np.maximum(x, 0.0) - x * z + np.log1p(np.exp(-np.abs(x)))


def objective(cfg, T):
    """[K, T] 0/1 objective rows (:974-976)"""
    return (np.arange(T)[None, :] < np.asarray(cfg["counts"])[:, None]).astype(F64)


def count_terms(P, cond, cfg):
    """The min-element count penalty of each image in fp64 on P [B,T]: the [B,K] sums, the [B,K] tie mask of reduce_min and
    the magnitudes of their terms.  cond [B,T] weighs the P / (1 - P) conditioning of log(1 - P) (0 where P is exact)."""
    T = P.shape[1]
    z = objective(cfg, T)[None]                                             # [1,K,T]
    x = logit_eps(P)[:, None, :]
    mx = (np.abs(np.log(P + 1e-8)) + np.abs(np.log(1 - P + 1e-8)) + 2 + cond * P / (1 - P + 1e-8))[:, None, :]
    sx = sigmoid64(x)
    bce = bce_logits(z, x).sum(-1)
    mag = (np.abs(x) * (1 + z) + np.log1p(np.exp(-np.abs(x))) + mx * np.abs(sx - z)).sum(-1)
    tied = bce <= bce.min(-1, keepdims=True) * (1 + 1e-12)
    return bce, tied, mag, sx, z, mx


def magnitudes(case, cfg, P=None, cond=None):
    """depth * sum|terms| of every output entry, in fp64 (see the module docstring)"""
    lo = case["lo"].astype(F64)
    B, T = lo.shape
    P = sigmoid64(lo) if P is None else P
    cond = np.ones_like(P) if cond is None else cond
    g = {k: abs(cfg.get(k, 0.0)) for k in GAMMAS}
    gp, gm = np.abs(case["gp"].astype(F64)), abs(float(case["gm"][0]))
    cs = float(cfg["canvas_size"])
    smin, smax = cfg.get("area_minmax", (0.0, 0.0))
    K = len(cfg["counts"])
    A = {}

    sp = lambda v: np.logaddexp(0.0, v)
    if g["gamma_num"] > 1e-8:
        ent = P * sp(-lo) + (1 - P) * sp(lo) + P * np.abs(lo)               # P |lo|: the rounding of P, seen through 1 - P
        A["pr_num"] = g["gamma_num"] * (T + 4) * ent.sum(-1)
        dlo = gp[:, None] * g["gamma_num"] * np.abs(lo) * P
    else:
        A["pr_num"] = np.zeros(B)
        dlo = np.zeros((B, T))
    A["num_min"], A["margin"] = np.zeros(B), np.zeros(1)
    if g["gamma_margin"] > 1e-8:
        bce, tied, mag, sx, z, mx = count_terms(P, cond, cfg)
        A["num_min"] = g["gamma_elem"] * (T + 4) * mag.max(-1)
        pb = pbar_of(case)
        mobj = objective(cfg, T).mean(0)
        xb = logit_eps(pb)
        mxb = np.abs(np.log(pb + 1e-8)) + np.abs(np.log(1 - pb + 1e-8)) + 2 + pb / (1 - pb + 1e-8)
        sb = sigmoid64(xb)
        A["margin"] = np.array([g["gamma_margin"] * (T + 4) * (np.abs(xb) * (1 + mobj) + np.log1p(np.exp(-np.abs(xb)))
                                                               + mxb * np.abs(sb - mobj)).sum()])
        pq = P * (1 - P)                   # P (1 - P) dlogit_eps(P) takes 1 - P from the same fp32 value twice: no conditioning
        pq_cond = P * (1 - P + cond * P)   # the margin's P (1 - P) alone: 1 - P carries the rounding of P
        n = tied.sum(-1)[:, None]
        sx_mag = sx + sx * (1 - sx) * mx                                    # sigmoid of the fp32 logit
        dx = (tied[:, :, None] * (sx_mag + z)).sum(1) / n
        dlo = dlo + gp[:, None] * g["gamma_elem"] * dx * dlogit_eps(P) * pq
        dlo = dlo + gm * g["gamma_margin"] * F64(case["inv_B"]) * (sb + mobj + sb * (1 - sb) * mxb) * dlogit_eps(pb) * pq_cond
    A["d_log_odds"] = (K + 6) * dlo

    sc, sh = case["sc"].astype(F64), case["sh"].astype(F64)
    px = sc * cs
    cx, cy = (sh[..., 0] + 1) * cs / 2, (sh[..., 1] + 1) * cs / 2
    mcx, mcy = (np.abs(sh[..., 0]) + 1) * cs / 2, (np.abs(sh[..., 1]) + 1) * cs / 2
    a_hi, a_lo = px - smin >= 0, smax - px >= 0
    A["area"] = (2 * T + 4) * ((smax + px) * a_lo + (px + smin) * a_hi).sum(-1) / T
    lx, ly = -(cx - px / 2) >= 0, -(cy - px / 2) >= 0
    hx, hy = cx + px / 2 - cs >= 0, cy + px / 2 - cs >= 0
    A["out"] = (4 * T + 4) * ((lx + hx) * (mcx + px / 2) + (ly + hy) * (mcy + px / 2) + (hx + hy) * cs).sum(-1)
    D = px[:, :, None] - px[:, None, :]
    s_act = np.abs(D) - 3 >= 0
    A["size"] = (T * T + 4) * (s_act * (px[:, :, None] + px[:, None, :] + 3)).sum((-1, -2))
    xd, yd = np.abs(cx[:, :, None] - cx[:, None, :]), np.abs(cy[:, :, None] - cy[:, None, :])
    v = (px[:, :, None] + px[:, None, :]) / 2 - np.maximum(xd, yd)
    o_act = (v >= 0) & ~np.eye(T, dtype=bool)[None]
    mpair = lambda m: m[:, :, None] + m[:, None, :]
    A["overlap"] = (T * T + 4) * (o_act * (mpair(px) / 2 + mpair(mcx) + mpair(mcy))).sum((-1, -2))
    A["per_image"] = (A["pr_num"] + A["num_min"] + g["gamma_area"] * A["area"] + g["gamma_bbox"] * (A["out"] + A["overlap"])
                      + g["gamma_size"] * A["size"]) * 2

    # geometry gradients: sum of |contributions| to d px, d cx, d cy; every entry accumulates at most 4 T + 6 of them
    gpt = gp[:, None]
    dpx = gpt * (g["gamma_area"] / T * (a_hi + a_lo) + g["gamma_bbox"] * 0.5 * (lx + ly + hx + hy)
                 + g["gamma_size"] * 2 * s_act.sum(-1) + g["gamma_bbox"] * o_act.sum(-1))
    xr = xd >= yd
    dcx = gpt * g["gamma_bbox"] * ((lx + hx) + 2 * (o_act & xr).sum(-1))
    dcy = gpt * g["gamma_bbox"] * ((ly + hy) + 2 * (o_act & ~xr).sum(-1))
    A["d_scales"] = (4 * T + 6) * dpx * cs
    A["d_shifts"] = (4 * T + 6) * np.stack([dcx, dcy], -1) * cs / 2
    return A


def excess(got, ref, mag, ulps=ULPS):
    """max of |got - ref| / (ulps * 2^-23 * mag + FLT_MIN); <= 1 passes, a NaN in got fails"""
    got = np.asarray(got, F64)
    err = np.abs(got - np.asarray(ref, F64)) / (ulps * EPS32 * np.asarray(mag, F64) + FLT_MIN)
    return float(np.nan_to_num(err, nan=np.inf).max()) if err.size else 0.0


def run_and_check(L, dev, case, cfg, ref=None, A=None):
    """Forward and backward of one case against the fp64 oracle under the per-entry bounds; components = NULL, g_margin =
    NULL (against g_margin = 0) and a second run give the same bits.  Returns the kernel's outputs and the oracle's."""
    d = to_dev(case, dev)
    ref = oracle(case, cfg) if ref is None else ref
    A = magnitudes(case, cfg) if A is None else A
    per_image, comps, margin = forward(L, d, case, cfg)
    out = {"per_image": np_(per_image), "margin": np_(margin)}
    out.update({k: np_(comps[:, i]) for i, k in enumerate(COMPONENTS)})
    assert excess(out["per_image"], ref["per_image"], A["per_image"]) <= 1.0
    assert excess(out["margin"], np.atleast_1d(ref["margin"]), A["margin"]) <= 1.0
    for k in COMPONENTS:
        assert excess(out[k], ref[k], A[k]) <= 1.0, k
    again = forward(L, d, case, cfg)
    plain = forward(L, d, case, cfg, components=False)
    for a, b in ((again[0], per_image), (again[1], comps), (again[2], margin), (plain[0], per_image), (plain[2], margin)):
        assert torch.equal(a, b)

    grads = backward(L, d, case, cfg)
    out.update(d_log_odds=np_(grads[0]), d_shifts=np_(grads[1]), d_scales=np_(grads[2]))
    for k in ("d_log_odds", "d_shifts", "d_scales"):
        assert excess(out[k], ref[k], A[k]) <= 1.0, k
    for a, b in zip(backward(L, d, case, cfg), grads):
        assert torch.equal(a, b)
    null_gm, zero_gm = backward(L, d, case, cfg, g_margin=None), backward(L, d, case, cfg, g_margin="zero")
    for a, b in zip(null_gm, zero_gm):
        assert torch.equal(a, b)
    return out, ref


# ---------------------------------------------------------------------------------------------------------------------
# inputs
# ---------------------------------------------------------------------------------------------------------------------
def host_psum(lo):
    return sigmoid64(lo.astype(F64)).sum(0).astype(F32)


def make_case(lo, sh, sc, gp, gm, psum=None, inv_B=None):
    lo = np.asarray(lo, F32)
    return dict(lo=lo, sh=np.asarray(sh, F32), sc=np.asarray(sc, F32), gp=np.asarray(gp, F32), gm=np.array([gm], F32),
                psum=host_psum(lo) if psum is None else np.asarray(psum, F32),
                inv_B=F32(1.0 / lo.shape[0]) if inv_B is None else F32(inv_B))


def near_ties(case, cfg, rel=2.0 ** -16, rel_count=2.0 ** -12):
    """[B] rows where a branch point of the geometry lies within ``rel`` of its operands' magnitude, or where the two smallest
    count penalties of distinct objectives (counts clipped to [0, T]) differ by less than ``rel_count`` of their magnitude:
    there fp32 and fp64 may take different sub-gradients.  Identical objectives tie exactly in both and are not flagged."""
    lo, sc, sh = (case[k].astype(F64) for k in ("lo", "sc", "sh"))
    B, T = lo.shape
    cs = float(cfg["canvas_size"])
    smin, smax = cfg.get("area_minmax", (0.0, 0.0))
    px = sc * cs
    cx, cy = (sh[..., 0] + 1) * cs / 2, (sh[..., 1] + 1) * cs / 2
    m = np.abs(cx) + np.abs(cy) + px + cs + abs(smin) + abs(smax)
    near = lambda q, mag: np.abs(q) < rel * mag
    bad = (near(px - smin, m) | near(smax - px, m) | near(cx - px / 2, m) | near(cy - px / 2, m)
           | near(cx + px / 2 - cs, m) | near(cy + px / 2 - cs, m)).any(-1)
    mp = m[:, :, None] + m[:, None, :]
    D = px[:, :, None] - px[:, None, :]
    dx, dy = cx[:, :, None] - cx[:, None, :], cy[:, :, None] - cy[:, None, :]
    v = (px[:, :, None] + px[:, None, :]) / 2 - np.maximum(np.abs(dx), np.abs(dy))
    off = ~np.eye(T, dtype=bool)[None]
    pair = near(np.abs(D) - 3, mp) | (off & (near(v, mp) | ((v > 0) & (near(np.abs(dx) - np.abs(dy), mp) | near(dx, mp) | near(dy, mp)))))
    bad |= pair.any((-1, -2))
    if cfg.get("gamma_margin", 0.0) > 1e-8:
        eff = sorted({min(max(c, 0), T) for c in cfg["counts"]})
        if len(eff) > 1:
            sub = dict(cfg, counts=eff)
            bce, _, mag, *_ = count_terms(sigmoid64(lo), np.ones_like(lo), sub)
            s = np.sort(bce, -1)
            bad |= (s[:, 1] - s[:, 0]) < rel_count * mag.max(-1)
    return bad


def random_case(B, T, cfg, seed, lo_sd=2.0, lo_max=7.0):
    """Non-dyadic inputs; rows near a branch point (near_ties) are drawn again."""
    rng = np.random.default_rng(seed)

    def draw(n):
        return (np.clip(rng.normal(0, lo_sd, (n, T)), -lo_max, lo_max), np.tanh(rng.normal(0, 0.8, (n, T, 2))),
                sigmoid64(rng.normal(-1.0, 0.6, (n, T))))

    lo, sh, sc = draw(B)
    case = make_case(lo, sh, sc, rng.normal(0, 1, B), 0.7)
    for _ in range(100):
        bad = near_ties(case, cfg)
        if not bad.any():
            break
        for k, a in zip(("lo", "sh", "sc"), draw(int(bad.sum()))):
            case[k][bad] = a.astype(F32)
    assert not near_ties(case, cfg).any()
    case["psum"] = host_psum(case["lo"])
    return case


# ---------------------------------------------------------------------------------------------------------------------
# 1. TF's tie rules, exact
# ---------------------------------------------------------------------------------------------------------------------
CS = 64
MINMAX = (10.0, 20.0)
# four boxes (centre x, centre y, size in pixels) well inside the canvas, sizes strictly inside the window, no two sizes
# 3 apart, no two boxes touching, no |dx| = |dy|
BASE = [(12, 12, 12), (44, 14, 13), (14, 46, 17), (46, 48, 19)]
TIE_CASES = {
    "size_min": [(12, 12, 10), (44, 14, 15), (14, 46, 17), (46, 48, 19)],          # px = size_min
    "size_max": [(12, 12, 12), (44, 14, 13), (14, 46, 18), (46, 48, 20)],          # px = size_max
    "edge_0": [(6, 12, 12), (44, 6.5, 13), (14, 46, 17), (46, 48, 19)],            # min x = 0, min y = 0
    "edge_cs": [(12, 12, 12), (57.5, 14, 13), (14, 55.5, 17), (46, 44, 19)],       # max x = 64, max y = 64
    "size_3": [(12, 12, 12), (44, 14, 15), (14, 46, 17), (46, 48, 19)],            # |12 - 15| = 3
    "touching": [(12, 12, 12), (24.5, 14, 13), (14, 46, 17), (46, 48, 19)],        # v = 0, xd = 12.5 > yd = 2
    "xd_eq_yd": [(12, 12, 12), (20, 20, 13), (14, 46, 17), (46, 48, 19)],          # xd = yd = 8 < 12.5
    # xd = yd = 0: both ordered pairs route to x with sgn(0) = 0.  Were sgn(0) taken as 1, the two pairs' contributions
    # (-g then +g, g = g_per_image * gamma_bbox) would still cancel exactly, so that choice is not observable
    "same_centre": [(12, 12, 12), (12, 12, 13), (14, 46, 17), (46, 48, 19)],
    # combined: a box at size_min touching the left edge and another box; two boxes at size_max 3 apart from a third
    # whose corners touch theirs (v = 0 at xd = yd); identical centres on the lower edge
    "combined_a": [(5, 12, 10), (15, 14, 10), (14, 46, 17), (46, 48, 19)],
    "combined_b": [(12, 12, 20), (28.5, 28.5, 13), (14, 46, 17), (46, 56.5, 15)],
    "combined_c": [(12, 6, 12), (12, 6, 12), (40, 46, 17), (46, 8, 16)],
}
TIE_KINDS = ("size_min", "size_max", "edge_0", "edge_cs", "size_3", "touching", "xd_eq_yd", "same_centre")


def ties_in(boxes):
    """which exact ties one row of (cx, cy, px) holds, in exact arithmetic"""
    found = set()
    for i, (cx, cy, p) in enumerate(boxes):
        found |= {"size_min"} if p == MINMAX[0] else set()
        found |= {"size_max"} if p == MINMAX[1] else set()
        found |= {"edge_0"} if 0 in (cx - p / 2, cy - p / 2) else set()
        found |= {"edge_cs"} if CS in (cx + p / 2, cy + p / 2) else set()
        for j, (ux, uy, q) in enumerate(boxes):
            if j == i:
                continue
            xd, yd = abs(cx - ux), abs(cy - uy)
            v = (p + q) / 2 - max(xd, yd)
            found |= {"size_3"} if abs(p - q) == 3 else set()
            found |= {"touching"} if v == 0 else set()
            if v >= 0 and xd == yd:
                found |= {"same_centre"} if xd == 0 else {"xd_eq_yd"}
    return found


def boxes_case(rows, lo, gp, gm=0.5):
    """(cx, cy, px) rows -> exact fp32 inputs at canvas 64: shift = 2 cx / 64 - 1, scale = px / 64"""
    b = np.asarray(rows, F64)
    sh = np.stack([2 * b[..., 0] / CS - 1, 2 * b[..., 1] / CS - 1], -1)
    case = make_case(lo, sh, b[..., 2] / CS, gp, gm)
    assert np.array_equal(case["sh"].astype(F64), sh) and np.array_equal(case["sc"].astype(F64), b[..., 2] / CS)
    return case


EXACT_CFG = dict(canvas_size=CS, counts=[1, 3], max_steps=4, gamma_num=0.5, gamma_margin=2.0, gamma_elem=0.75,
                 gamma_bbox=1.5, gamma_size=0.25, gamma_area=2.0, area_minmax=MINMAX)


@pytest.mark.parametrize("name", list(TIE_CASES))
def test_tie_rules_exact(cuda_device, name):
    """Each tie of TF's sub-gradient rules on its own (and three rows that combine several): max(v, 0) passes the gradient at
    v = 0 (size window, canvas edges, pairwise size, touching boxes), maximum(xd, yd) routes to xd when xd = yd, abs'(0) = 0
    for identical centres.  Geometry values and gradients bit-equal to the fp64 oracle; the rest within the bounds."""
    L = _lib.load()
    rows = TIE_CASES[name]
    found = ties_in(rows)
    if name.startswith("combined"):
        assert len(found) >= 2, found
    else:
        assert found == {name}, found
    assert ties_in(BASE) == set()
    # row 0: the tie; row 1: the same boxes in reverse order (the other member of each pair comes first); row 2: the tie-free
    # base layout
    case = boxes_case([rows, rows[::-1], BASE], lo=[[1.5, -0.5, 2.25, -3.0]] * 3, gp=[0.75, -1.25, 0.5])
    out, ref = run_and_check(L, cuda_device, case, EXACT_CFG)
    for k in ("area", "out", "size", "overlap", "d_shifts", "d_scales"):
        assert np.array_equal(out[k].astype(F64), ref[k]), k


# reduce_min splits the gradient equally among tied counts; (counts, T, log-odds of one row)
SPLIT_CASES = {
    "duplicated_3_3": ([3, 3], 4, [1.5, -0.5, 2.0, -2.5]),
    "above_T_3_4_at_T3": ([3, 4], 3, [1.5, -0.5, 2.0]),
    "above_T_1_3_at_T1": ([1, 3], 1, [-1.25]),
    "three_way_2_5_7_at_T2": ([2, 5, 7], 2, [0.75, 2.5]),
    "three_way_with_a_loser": ([4, 0, 4, 4], 4, [1.5, 2.0, -0.5, 3.0]),
    "distinct_rows_at_P_half": ([1, 2], 2, [1.5, 0.0]),      # objectives [1, 0] and [1, 1] tie where P = 0.5 exactly
}


@pytest.mark.parametrize("name", list(SPLIT_CASES))
def test_min_element_split(cuda_device, name):
    """The min-element penalty at exact ties of reduce_min: num_min and d_log_odds against fp64 within the bounds, with the
    gradient of the count penalty split equally among the tied counts (the margin term kept small beside it)."""
    L = _lib.load()
    counts, T, lo = SPLIT_CASES[name]
    cfg = dict(canvas_size=CS, counts=counts, max_steps=T, gamma_margin=0.125, gamma_elem=4.0, gamma_num=0.25,
               gamma_bbox=1.0, gamma_size=0.5, gamma_area=0.5, area_minmax=MINMAX)
    rows = np.asarray(BASE[:T], F64)
    case = boxes_case([rows, rows], lo=[lo, [-v for v in lo]], gp=[0.75, -0.5], gm=1.0)
    _, tied, *_ = count_terms(sigmoid64(case["lo"].astype(F64)), np.ones((2, T)), cfg)
    assert tied.sum(-1)[0] >= 2                                             # row 0 holds the tie; row 1 has the log-odds negated
    run_and_check(L, cuda_device, case, cfg)


# ---------------------------------------------------------------------------------------------------------------------
# 2. gates
# ---------------------------------------------------------------------------------------------------------------------
ALL_ON = dict(gamma_num=0.7, gamma_margin=3.0, gamma_elem=2.0, gamma_bbox=1.5, gamma_size=0.5, gamma_area=0.25)
GATES = {
    "elem_without_margin": dict(ALL_ON, gamma_margin=0.0, gamma_num=0.0),   # :973 gates both count penalties on gamma_margin
    "margin_without_elem": dict(ALL_ON, gamma_elem=0.0),
    "num_below_gate": dict(ALL_ON, gamma_num=1e-9),
    **{f"{k}_alone": {k: ALL_ON[k]} for k in GAMMAS if k != "gamma_elem"},
}


@pytest.mark.parametrize("name", list(GATES))
def test_gates(cuda_device, name):
    """gamma_margin = 0 turns off num_min, margin and every log-odds gradient even with gamma_elem > 0; gamma_margin > 0
    with gamma_elem = 0 keeps the margin; gamma_num <= 1e-8 gives pr_num exactly 0; each gamma alone, so that every
    component's value and gradient is compared on its own."""
    L = _lib.load()
    cfg = dict(canvas_size=50, counts=[1, 3], max_steps=4, area_minmax=(11.0, 15.0), **GATES[name])
    case = random_case(129, 4, cfg, seed=len(name))
    out, ref = run_and_check(L, cuda_device, case, cfg)
    g = GATES[name]
    if g.get("gamma_margin", 0.0) == 0.0:
        assert np.all(out["num_min"] == 0) and np.all(out["margin"] == 0)
        if g.get("gamma_num", 0.0) == 0.0:
            assert np.all(out["d_log_odds"] == 0)
    else:
        assert out["margin"][0] != 0
    if g.get("gamma_elem", 0.0) == 0.0:
        assert np.all(out["num_min"] == 0)
    if g.get("gamma_num", 0.0) <= 1e-8:
        assert np.all(out["pr_num"] == 0)
    if not any(g.get(k, 0.0) for k in ("gamma_bbox", "gamma_size", "gamma_area")):
        assert np.all(out["d_shifts"] == 0) and np.all(out["d_scales"] == 0)


# ---------------------------------------------------------------------------------------------------------------------
# 3. limits
# ---------------------------------------------------------------------------------------------------------------------
LIMITS = [
    pytest.param(1, [0, 1, 3], 1, 50, id="T1-K3-B1"),
    pytest.param(2, [1, 3], 127, 50, id="T2-K2-B127"),
    pytest.param(7, [0, 2, 3, 5, 7, 8, 9, 12], 128, 50, id="T7-K8-B128"),
    pytest.param(16, [16, 3, 20], 129, 64, id="T16-K3-B129"),
    pytest.param(16, [0, 1, 2, 4, 6, 9, 13, 17], 4097, 50, id="T16-K8-B4097"),
    pytest.param(7, [4], 4097, 64, id="T7-K1-B4097"),
]


@pytest.mark.parametrize("T,counts,B,cs", LIMITS)
def test_limits(cuda_device, T, counts, B, cs):
    """T from 1 to MOG_ASR_MAX_STEPS, 1 to MOG_ASR_MAX_COUNTS counts (a count of 0, counts above T), batch sizes around the
    128-thread block, non-dyadic inputs at canvas 50 and 64: every entry within the bounds, the margin written (by one thread)
    and right at every B."""
    assert T <= _lib.MOG_ASR_MAX_STEPS and len(counts) <= _lib.MOG_ASR_MAX_COUNTS
    L = _lib.load()
    cfg = dict(canvas_size=cs, counts=counts, max_steps=T, area_minmax=(11.0, 15.0), **ALL_ON)
    case = random_case(B, T, cfg, seed=T * 1000 + B)
    out, ref = run_and_check(L, cuda_device, case, cfg)
    assert np.isfinite(out["margin"]).all() and out["margin"][0] > 0


# ---------------------------------------------------------------------------------------------------------------------
# 4. the column sum past one grid pass
# ---------------------------------------------------------------------------------------------------------------------
def colsum_pass(dev):   # mog_asr_reg_colsum: 4 CTAs per SM x 256 threads, one row per thread
    return torch.cuda.get_device_properties(dev).multi_processor_count * 4 * 256


@pytest.mark.parametrize("T", [1, 16])
def test_colsum_past_one_pass(cuda_device, T):
    """psum[t] += sum_b sigmoid(log_odds[b][t]) over about 2.5 grid passes and a ragged remainder, onto a non-zero psum.
    The sum ends in one atomic add per warp and is not bit-deterministic, so it is held to fp64 within the bound of its
    summation depth: sigmoid, the rows of one thread, five warp-shuffle levels, then the atomics of every warp in turn, all
    of positive terms."""
    L = _lib.load()
    dev = cuda_device
    per_pass = colsum_pass(dev)
    B = 5 * per_pass // 2 + 1237
    assert B > 2 * per_pass and B % 256 != 0
    rng = np.random.default_rng(T)
    lo = rng.normal(0, 3, (B, T)).astype(F32)
    init = rng.uniform(0.5, 2.0, T).astype(F32) * B / 4
    psum = torch.from_numpy(init).to(dev)
    call(L.mog_asr_reg_colsum, ptr(torch.from_numpy(lo).to(dev)), ptr(psum), B, T)
    ref = init.astype(F64) + sigmoid64(lo.astype(F64)).sum(0)
    rows = -(-B // per_pass)
    warps = per_pass // 32
    depth = 3 + rows + 5 + warps
    assert excess(np_(psum), ref, depth * ref, ulps=2) <= 1.0


# ---------------------------------------------------------------------------------------------------------------------
# 5. the data-parallel contract on one GPU
# ---------------------------------------------------------------------------------------------------------------------
def test_data_parallel_shards(cuda_device):
    """Shards of 100 and 157 images: psum of each by colsum, added on the device as an all-reduce would; forward and backward
    of each shard with that psum and inv_global_batch = 1/257 give, concatenated, the bits of the whole-batch call with the
    same psum, the same margin on every shard, and both match the oracle with the global batch mean."""
    L = _lib.load()
    dev = cuda_device
    T = 6
    cfg = dict(canvas_size=50, counts=[1, 2, 4], max_steps=T, area_minmax=(11.0, 15.0), **ALL_ON)
    whole = random_case(257, T, cfg, seed=257)
    parts = [slice(0, 100), slice(100, 257)]
    psum = torch.zeros(T, device=dev)
    for s in parts:
        p = torch.zeros(T, device=dev)
        call(L.mog_asr_reg_colsum, ptr(torch.from_numpy(np.ascontiguousarray(whole["lo"][s])).to(dev)), ptr(p), s.stop - s.start, T)
        psum += p
    ref_psum = sigmoid64(whole["lo"].astype(F64)).sum(0)
    assert excess(np_(psum), ref_psum, (3 + 1 + 5 + 8) * ref_psum, ulps=2) <= 1.0
    whole["psum"], whole["inv_B"] = np_(psum), F32(1.0 / 257)
    out, ref = run_and_check(L, dev, whole, cfg)
    for s in parts:
        shard = {k: (whole[k][s] if k in ("lo", "sh", "sc", "gp") else whole[k]) for k in whole}
        A = {k: (v[s] if k not in ("margin",) else v) for k, v in magnitudes(whole, cfg).items()}
        sref = {k: (v[s] if np.ndim(v) else v) for k, v in ref.items()}
        sout, _ = run_and_check(L, dev, shard, cfg, ref=sref, A=A)
        assert np.array_equal(sout["margin"], out["margin"])
        for k in ("per_image", *COMPONENTS, "d_log_odds", "d_shifts", "d_scales"):
            assert np.array_equal(sout[k], out[k][s]), k


# ---------------------------------------------------------------------------------------------------------------------
# 6. confident z_pres
# ---------------------------------------------------------------------------------------------------------------------
def p32(lo, ulp=0):
    """fl(1 / fl(1 + fl(exp(-lo)))) with exp(-lo) moved by ``ulp`` units in the last place"""
    e = np.exp(-lo.astype(F64)).astype(F32)
    for _ in range(abs(ulp)):
        e = np.nextafter(e, F32(np.inf) if ulp > 0 else F32(0))
    return (F32(1) / (F32(1) + e)).astype(F32)


def fp32p_reference(case, cfg, P):
    """The header's formulas in fp64, on the fp32 P the kernel computes: pr_num, num_min, margin, d_log_odds"""
    lo = case["lo"].astype(F64)
    T = lo.shape[1]
    gp, gm = case["gp"].astype(F64)[:, None], F64(case["gm"][0])
    gn, gmar, ge = cfg["gamma_num"], cfg["gamma_margin"], cfg["gamma_elem"]
    sp = lambda v: np.logaddexp(0.0, v)
    r = {"pr_num": (gn * (P * sp(-lo) + (1 - P) * sp(lo))).sum(-1)}
    bce, tied, _, sx, z, _ = count_terms(P, np.zeros_like(P), cfg)
    r["num_min"] = ge * bce.min(-1)
    pb = (case["psum"] * case["inv_B"]).astype(F64)                          # one fp32 rounding, as in the kernel
    mobj = objective(cfg, T).mean(0)
    xb = logit_eps(pb)
    r["margin"] = np.array([gmar * bce_logits(mobj, xb).sum()])
    dx = (tied[:, :, None] * (sx - z)).sum(1) / tied.sum(-1)[:, None]
    dP = gp * ge * dx * dlogit_eps(P) + gm * gmar * (sigmoid64(xb) - mobj) * dlogit_eps(pb) * F64(case["inv_B"])
    r["d_log_odds"] = gp * gn * (-lo * P * (1 - P)) + dP * P * (1 - P)
    return r


def test_confident_zpres(cuda_device):
    """Log-odds up to +-30 with pr_num and both count penalties on.  Reference: the header's formulas in fp64 on the fp32 P
    emulated on the host; where P >= 1/2 every input is picked so that +-2 ulp of expf cannot change that P (asserted), below
    1/2 the P / (1 - P) conditioning is below 1 and enters the bound.  Where P rounds to 1.0f (log-odds >= 17.5) d_log_odds
    is exactly 0 and num_min uses logit_eps(1.0f); no output is NaN or Inf."""
    L = _lib.load()
    grid = np.arange(-240, 241, dtype=F64) / 8
    P_all = p32(grid.astype(F32))
    steady = np.all([p32(grid.astype(F32), u) == P_all for u in (-2, -1, 1, 2)], 0)
    pick = grid[(grid < 0) | steady]
    rng = np.random.default_rng(6)
    B, T = 256, 4
    cond_ = lambda lo: (lo < 0).astype(F64)
    cfg = dict(canvas_size=50, counts=[1, 3], max_steps=T, gamma_num=0.7, gamma_margin=3.0, gamma_elem=2.0)

    def near_tie(lo):    # the two counts' penalties within 1e-3 of their magnitude: fp32 and fp64 may pick different ones
        bce, _, mag, *_ = count_terms(p32(lo).astype(F64), cond_(lo), cfg)
        return np.abs(bce[:, 0] - bce[:, 1]) <= 1e-3 * mag.max(-1)

    lo = rng.choice(pick, (B, T)).astype(F32)
    lo[:8] = np.array([[30, 17.5, 20, 25], [-30, -17.5, 17.5, 30], [8, 10, 12, 15], [-8, -12, 16, 16.5]] * 2, F32)
    for _ in range(100):
        redo = near_tie(lo)
        if not redo.any():
            break
        lo[redo] = rng.choice(pick, (int(redo.sum()), T))
    assert not near_tie(lo).any() and lo[0, 0] == 30 and lo[7, 3] == 16.5
    P = p32(lo)
    assert np.all([np.array_equal(p32(lo[lo >= 0], u), P[lo >= 0]) for u in (-2, -1, 1, 2)])
    assert (lo >= 17.5).any() and np.all(P[lo >= 17.5] == 1) and np.all(P[lo < 16.5] < 1)
    cond = cond_(lo)
    case = boxes_case([BASE[:T]] * B, lo=lo, gp=rng.normal(0, 1, B), gm=0.7)

    d = to_dev(case, cuda_device)
    per_image, comps, margin = forward(L, d, case, cfg)
    d_lo, d_sh, d_sc = backward(L, d, case, cfg)
    for t in (per_image, comps, margin, d_lo, d_sh, d_sc):
        assert torch.isfinite(t).all()
    ref = fp32p_reference(case, cfg, P.astype(F64))
    A = magnitudes(case, cfg, P=P.astype(F64), cond=cond)
    got = {"pr_num": np_(comps[:, 0]), "num_min": np_(comps[:, 1]), "margin": np_(margin), "d_log_odds": np_(d_lo)}
    for k, v in got.items():
        assert excess(v, ref[k], A[k]) <= 1.0, k
    assert excess(np_(per_image), ref["pr_num"] + ref["num_min"], A["pr_num"] + A["num_min"]) <= 1.0
    assert np.all(np_(d_lo)[P == 1] == 0)
    # a row saturated at every step: each bce is that of logit_eps(1.0f) = log(1 + 1e-8) - log(1e-8)
    x1 = float(np.log(F32(1) + F32(1e-8)) - np.log(F32(1e-8)))
    assert abs(x1 - 18.420681) < 1e-5
    sat = np.all(P == 1, -1)
    assert sat.any()
    z = objective(cfg, T)
    want = cfg["gamma_elem"] * min(bce_logits(z[k], x1).sum() for k in range(len(cfg["counts"])))
    assert np.all(np.abs(np_(comps[:, 1])[sat] - want) <= 8 * EPS32 * want)
