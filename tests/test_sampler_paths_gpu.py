"""GPU parity of the sampler's other forms -- the fused write + composite, the (s, x, y) entry points and the batched
(``u_batch_div > 1``) backward -- against the fp64 oracle, one case per backward dispatch class.

``launch_bwd`` (csrc/mog_stn.cu) sends every backward call to one of these instantiations, by source width, by whether the
output is at least as large as the source, and by how dU outside the footprint is zeroed (``coop_zero``: 0 each warp its own
image, 1 the CTA sweeps its group of images, 2 the bulk-copy engine).  Each case below names the class it reaches.  Every
output buffer is pre-filled with NaN through the C ABI, so an element a kernel never writes fails the comparison.

Tolerances are the stated ones (DESIGN.md section 4): forwards bit-exact; gradients within ``GRAD_RTOL`` of the fp64 oracle
relative to the sum of |terms| entering each entry."""
import numpy as np
import pytest
import torch

from mog_asr_b200 import _lib, synth
from oracle import stn_ref_numpy as R
from tests import helpers as H

pytestmark = pytest.mark.gpu

THRESHOLD = np.float32(0.9)

# (source, output) sizes -- for the composite (window, canvas) -- and the backward class launch_bwd picks for them
CLASSES = [
    pytest.param(28, 50, id="28to50"),       # stn_bwd_col_kernel<., 1>
    pytest.param(64, 256, id="64to256"),     # stn_bwd_col_kernel<., 2>, float2 pair stores
    pytest.param(63, 127, id="63to127"),     # stn_bwd_col_kernel<., 2>, odd Ws: scalar stores
    pytest.param(28, 20, id="28to20"),       # stn_bwd_warp_kernel<., 1>, coop_zero = 0 (output smaller than the source)
    pytest.param(64, 50, id="64to50"),       # stn_bwd_warp_kernel<., 2>, coop_zero = 0
    pytest.param(96, 128, id="96to128"),     # stn_bwd_warp_kernel<., 4>, coop_zero = 2 (bulk zero; Ws > 64 streams)
    pytest.param(150, 160, id="150to160"),   # stn_bwd_warp_kernel<., 4>, coop_zero = 2, full cover: two strips
]

# theta kinds mixed into every batch, in this order (cycled); for the composite, z_pres (None: uniform in (0, 1)) and stop_sum
# below, exactly at or above the threshold go with them (the second nine images of a batch pair them differently)
KINDS = ("prior", "full", "corner", "outside", "flip_y", "full", "general", "prior", "flip_xy")
Z_PRES = (None, None, -0.7, None, 0.0, None, None, -0.7, None)
STOP_SUM = (1.3, THRESHOLD, 0.25, 0.25, 0.25, 0.25, 0.25, 0.25, 0.25)


def batch_size(src, dst):
    return 9 if max(src, dst) >= 128 else 18


def make_thetas(B, write, seed, general=True):
    """[B, 6] float32 thetas cycling through KINDS: read ([[s,0,x],[0,s,y]]) or write ([[1/s,0,-x/s],[0,1/s,-y/s]]) form of
    prior-like and full-cover (s, x, y); a footprint hanging over a corner; a footprint entirely out of range; t4 < 0 (the
    descending stream order) alone and with t0 < 0; a rotated and sheared theta (t01, t10 != 0).  general=False replaces
    the last by a full-cover theta (a batch without atomics in the backward)."""
    build = R.theta_write if write else R.theta_read
    sp, xp, yp = synth.sxy_prior_like(B, seed=seed)
    sf, xf, yf = synth.sxy_full_cover(B, seed=seed + 1)
    prior = build(sp, xp, yp).reshape(B, 6)
    full = build(sf, xf, yf).reshape(B, 6)
    corner = build(np.float32([0.3]), np.float32([0.9]), np.float32([-0.9])).reshape(6)
    th = np.empty((B, 6), np.float32)
    for b in range(B):
        kind = KINDS[b % len(KINDS)]
        if kind == "general" and not general:
            kind = "full"
        if kind == "prior":
            th[b] = prior[b]
        elif kind == "full":
            th[b] = full[b]
        elif kind == "corner":
            th[b] = corner
        elif kind == "outside":
            th[b] = [0.5, 0.0, 5.0, 0.0, 0.5, 5.0]
        elif kind in ("flip_y", "flip_xy"):
            th[b] = full[b]
            th[b, 4] = -th[b, 4]
            if kind == "flip_xy":
                th[b, 0] = -th[b, 0]
        else:
            th[b] = general_affine(full[b])
    return th


def general_affine(theta):
    """theta with its linear part rotated by 0.3 rad and sheared: t01, t10 != 0"""
    c, s = np.cos(0.3), np.sin(0.3)
    A = theta.reshape(2, 3)[:, :2].astype(np.float64) @ np.array([[c, -s], [s, c]]) @ np.array([[1.0, 0.2], [0.0, 1.0]])
    return np.concatenate([A, theta.reshape(2, 3)[:, 2:]], 1).reshape(6).astype(np.float32)


def separable(th):
    return (th[:, 1] == 0) & (th[:, 3] == 0)


def nan_buffer(shape, dev):
    return torch.full(shape, float("nan"), device=dev)


def ptr(t):
    return t.data_ptr() if t is not None else None


def call(fn, *args):
    rc = fn(*args)
    torch.cuda.synchronize()
    assert rc == 0, _lib.last_error()


def dz_reference(U, th, out_size, gcanvas, mask):
    """d loss / d z_pres in fp64 and the sum of |terms| entering it: dz[b] = m[b] * sum_n g[n] * sum_k w_k[n] I_k[n], the
    weights formed from the fp32 coordinates as in R.transformer_backward.  Out of range on an axis the tap pairs cancel
    exactly here and are skipped by the kernels (DESIGN.md "borders"), so only pixels in range on both axes count towards
    the magnitude."""
    full = R.transformer_full(U[..., None], th, out_size)
    B = U.shape[0]
    g = np.asarray(gcanvas, np.float64).reshape(B, -1)
    x, y = full["x"].astype(np.float64), full["y"].astype(np.float64)
    x0, x1, y0, y1 = (full[k].astype(np.float64) for k in ("x0", "x1", "y0", "y1"))
    w = ((x1 - x) * (y1 - y), (x1 - x) * (y - y0), (x - x0) * (y1 - y), (x - x0) * (y - y0))
    I = [full[k][..., 0].astype(np.float64) for k in ("Ia", "Ib", "Ic", "Id")]
    win = sum(wk * Ik for wk, Ik in zip(w, I))
    inside = (full["x0"] != full["x1"]) & (full["y0"] != full["y1"])
    absterms = np.where(inside, sum(np.abs(wk) * np.abs(Ik) for wk, Ik in zip(w, I)), 0.0)
    m = np.asarray(mask, np.float64)
    return m * (g * win).sum(1), (np.abs(g) * absterms).sum(1)


# ---------------------------------------------------------------------------------------------------------------------
# fused write + composite, theta given
# ---------------------------------------------------------------------------------------------------------------------
def composite_inputs(ws, cs, seed, general=True):
    """window, theta, z_pres, stop_sum, canvas, gcanvas for a batch mixing every theta kind with stop_sum below, exactly at
    and above the threshold and z_pres in (0, 1), 0 and negative.  Canvases hold no -0.0 (the in-place form skips canvas + 0)."""
    B = batch_size(ws, cs)
    rng = np.random.default_rng(seed)
    W = rng.random((B, ws, ws), dtype=np.float32)
    th = make_thetas(B, True, seed, general)
    z = rng.uniform(0.05, 0.95, B).astype(np.float32)
    stop = np.empty(B, np.float32)
    for b in range(B):
        k = (b + 4 * (b // len(KINDS))) % len(KINDS)
        if Z_PRES[k] is not None:
            z[b] = Z_PRES[k]
        stop[b] = STOP_SUM[k]
    canvas = rng.uniform(0.01, 1.0, (B, cs, cs)).astype(np.float32)
    g = rng.standard_normal((B, cs, cs), dtype=np.float32)
    return W, th, z, stop, canvas, g


@pytest.mark.parametrize("ws,cs", CLASSES)
@pytest.mark.parametrize("with_stop", [True, False], ids=["stop", "nostop"])
def test_write_composite_matches_the_oracle(cuda_device, ws, cs, with_stop):
    """mog_stn_write_composite_forward / _backward: the forward out of place and in place bit-exact with the oracle (inactive
    images untouched in place); dU, dtheta and dz within tolerance of the fp64 oracle; exactly zero gradients for inactive
    images; each gradient requested alone equal to the same gradient requested with the others."""
    L = _lib.load()
    dev = cuda_device
    W, th, z, stop, canvas, g = composite_inputs(ws, cs, seed=ws * 1000 + cs)
    B = W.shape[0]
    if not with_stop:
        stop = None
    mask = np.ones(B, bool) if stop is None else stop < THRESHOLD
    Wd, thd, zd, cd, gd = (torch.tensor(a, device=dev) for a in (W, th, z, canvas, g))
    sd = torch.tensor(stop, device=dev) if stop is not None else None
    thr = float(THRESHOLD)

    out = nan_buffer((B, cs, cs), dev)
    call(L.mog_stn_write_composite_forward, ptr(Wd), ptr(thd), ptr(zd), ptr(sd), thr, ptr(cd), ptr(out), B, ws, ws, cs, cs, None)
    ref = R.write_composite(canvas, W, th, z, mask)
    assert H.same_bits_or_nan(out.cpu().numpy(), ref)
    inplace = cd.clone()
    call(L.mog_stn_write_composite_forward, ptr(Wd), ptr(thd), ptr(zd), ptr(sd), thr, ptr(inplace), ptr(inplace), B, ws, ws, cs, cs,
         None)
    assert torch.equal(inplace, out)
    assert np.array_equal(inplace.cpu().numpy()[~mask].view(np.uint32), canvas[~mask].view(np.uint32))

    def backward(want_dU=True, want_dth=True, want_dz=True):
        dU = nan_buffer((B, ws, ws), dev) if want_dU else None
        dth = nan_buffer((B, 6), dev) if want_dth else None
        dz = nan_buffer((B,), dev) if want_dz else None
        call(L.mog_stn_write_composite_backward, ptr(Wd), ptr(thd), ptr(zd), ptr(sd), thr, ptr(gd), ptr(dU), ptr(dth), ptr(dz),
             B, ws, ws, cs, cs, None)
        return dU, dth, dz

    dU, dth, dz = backward()
    rU, rth, _ = R.write_composite_backward(W, th, z, mask, g)
    gwin = (mask * z.astype(np.float64))[:, None, None] * g
    aU, ath = R.backward_term_magnitudes(W[..., None], th, (cs, cs), gwin[..., None])
    rz, az = dz_reference(W, th, (cs, cs), g, mask)
    dU_, dth_, dz_ = dU.cpu().numpy(), dth.cpu().numpy(), dz.cpu().numpy()
    assert H.grad_excess(dU_, rU, aU[..., 0]) <= 1.0
    assert H.grad_excess(dth_.reshape(-1, 2, 3), rth, ath) <= 1.0
    assert H.grad_excess(dz_, rz, az) <= 1.0
    assert np.all(dU_[~mask] == 0) and np.all(dth_[~mask] == 0) and np.all(dz_[~mask] == 0)

    # one gradient at a time: the same bits (dU of a general-affine image is summed by atomics, in no fixed order)
    sep = torch.tensor(separable(th), device=dev)
    assert torch.equal(backward(True, False, False)[0][sep], dU[sep])
    assert torch.equal(backward(False, True, False)[1], dth)
    assert torch.equal(backward(False, False, True)[2], dz)


@pytest.mark.parametrize("ws,cs", CLASSES)
def test_write_composite_backward_is_deterministic_on_separable_batches(cuda_device, ws, cs):
    """Without a general-affine theta the composite backward has no atomics: two runs give the same bits."""
    L = _lib.load()
    dev = cuda_device
    W, th, z, stop, canvas, g = composite_inputs(ws, cs, seed=ws * 1000 + cs + 1, general=False)
    B = W.shape[0]
    Wd, thd, zd, sd, gd = (torch.tensor(a, device=dev) for a in (W, th, z, stop, g))
    runs = []
    for _ in range(2):
        bufs = [nan_buffer((B, ws, ws), dev), nan_buffer((B, 6), dev), nan_buffer((B,), dev)]
        call(L.mog_stn_write_composite_backward, ptr(Wd), ptr(thd), ptr(zd), ptr(sd), float(THRESHOLD), ptr(gd), *map(ptr, bufs),
             B, ws, ws, cs, cs, None)
        runs.append(bufs)
    for a, b in zip(*runs):
        assert torch.equal(a, b)


# ---------------------------------------------------------------------------------------------------------------------
# (s, x, y) entry points
# ---------------------------------------------------------------------------------------------------------------------
def sxy_inputs(B, seed):
    """(s, x, y) with s in {0.05, prior-like, 1.7, negative (descending stream)} plus a full-cover, a corner and an
    out-of-range footprint."""
    s, x, y = synth.sxy_prior_like(B, seed=seed)
    sf, xf, yf = synth.sxy_full_cover(B, seed=seed + 1)
    for b in range(B):
        k = b % 7
        if k == 1:
            s[b] = 0.05
        elif k == 2:
            s[b] = 1.7
        elif k == 3:
            s[b], x[b], y[b] = -sf[b], xf[b], yf[b]
        elif k == 4:
            s[b], x[b], y[b] = sf[b], xf[b], yf[b]
        elif k == 5:
            s[b], x[b], y[b] = 0.3, 0.9, -0.9
        elif k == 6:
            s[b], x[b], y[b] = 0.5, 5.0, 5.0
    return s, x, y


def sxy_chain_rule(dth, ath, s, x, y, write, g_shift_in, g_scale_in):
    """d_shift [B, 2], d_scale [B] from dtheta [B, 2, 3] by the fp64 chain rule of theta_read / theta_write, with the add-ins,
    and their sums of |terms|."""
    s, x, y = (np.asarray(v, np.float64) for v in (s, x, y))
    d00, d02, d11, d12 = dth[:, 0, 0], dth[:, 0, 2], dth[:, 1, 1], dth[:, 1, 2]
    a00, a02, a11, a12 = ath[:, 0, 0], ath[:, 0, 2], ath[:, 1, 1], ath[:, 1, 2]
    if not write:
        ds, dx, dy = d00 + d11, d02, d12
        ads, adx, ady = a00 + a11, a02, a12
    else:
        ds = ((x * d02 + y * d12) - (d00 + d11)) / s ** 2
        dx, dy = -d02 / s, -d12 / s
        ads = (np.abs(x) * a02 + np.abs(y) * a12 + a00 + a11) / s ** 2
        adx, ady = a02 / np.abs(s), a12 / np.abs(s)
    gsh, gsc = np.asarray(g_shift_in, np.float64), np.asarray(g_scale_in, np.float64)
    d_shift = np.stack([dx + gsh[:, 0], dy + gsh[:, 1]], 1)
    a_shift = np.stack([adx + np.abs(gsh[:, 0]), ady + np.abs(gsh[:, 1])], 1)
    return d_shift, ds + gsc, a_shift, ads + np.abs(gsc)


@pytest.mark.parametrize("src,dst", CLASSES)
def test_read_sxy_matches_the_oracle(cuda_device, src, dst):
    """mog_stn_read_sxy_forward / _backward: the glimpse bit-exact with the oracle on theta_read(s, x, y); dU, d_shift and
    d_scale (with non-zero add-ins) within tolerance of the fp64 oracle; the dU-less call gives the same d_shift / d_scale."""
    L = _lib.load()
    dev = cuda_device
    B = batch_size(src, dst)
    rng = np.random.default_rng(src * 1000 + dst + 7)
    s, x, y = sxy_inputs(B, seed=src + dst)
    U = rng.random((B, src, src), dtype=np.float32)
    g = rng.standard_normal((B, dst, dst), dtype=np.float32)
    g_shift_in = rng.standard_normal((B, 2), dtype=np.float32)
    g_scale_in = rng.standard_normal(B, dtype=np.float32)
    shd, scd = torch.tensor(np.stack([x, y], 1), device=dev), torch.tensor(s, device=dev)
    Ud, gd, gshd, gscd = (torch.tensor(a, device=dev) for a in (U, g, g_shift_in, g_scale_in))
    th = R.theta_read(s, x, y).reshape(B, 6)

    out = nan_buffer((B, dst, dst), dev)
    call(L.mog_stn_read_sxy_forward, ptr(Ud), ptr(shd), ptr(scd), ptr(out), B, src, src, dst, dst, None)
    assert H.same_bits_or_nan(out.cpu().numpy(), R.transformer(U[..., None], th, (dst, dst))[..., 0])

    def backward(want_dU):
        dU = nan_buffer((B, src, src), dev) if want_dU else None
        d_shift, d_scale = nan_buffer((B, 2), dev), nan_buffer((B,), dev)
        call(L.mog_stn_read_sxy_backward, ptr(Ud), ptr(shd), ptr(scd), ptr(gd), ptr(gshd), ptr(gscd), ptr(dU), ptr(d_shift),
             ptr(d_scale), B, src, src, dst, dst, None)
        return dU, d_shift, d_scale

    dU, d_shift, d_scale = backward(True)
    rU, rth = R.transformer_backward(U[..., None], th, (dst, dst), g[..., None])
    aU, ath = R.backward_term_magnitudes(U[..., None], th, (dst, dst), g[..., None])
    r_shift, r_scale, a_shift, a_scale = sxy_chain_rule(rth, ath, s, x, y, False, g_shift_in, g_scale_in)
    assert H.grad_excess(dU.cpu().numpy(), rU[..., 0], aU[..., 0]) <= 1.0
    assert H.grad_excess(d_shift.cpu().numpy(), r_shift, a_shift) <= 1.0
    assert H.grad_excess(d_scale.cpu().numpy(), r_scale, a_scale) <= 1.0
    _, d_shift2, d_scale2 = backward(False)
    assert torch.equal(d_shift2, d_shift) and torch.equal(d_scale2, d_scale)


@pytest.mark.parametrize("ws,cs", CLASSES)
def test_write_composite_sxy_matches_the_oracle(cuda_device, ws, cs):
    """mog_stn_write_composite_sxy_forward / _backward: the canvas bit-exact with the oracle on theta_write(s, x, y), out of
    place and in place; dU, dz, d_shift and d_scale (with non-zero add-ins) within tolerance of the fp64 oracle; inactive
    images get exactly the add-ins and zero dU / dz."""
    L = _lib.load()
    dev = cuda_device
    W, _, z, stop, canvas, g = composite_inputs(ws, cs, seed=ws * 1000 + cs + 2)
    B = W.shape[0]
    rng = np.random.default_rng(ws + cs)
    s, x, y = sxy_inputs(B, seed=ws * 3 + cs)
    g_shift_in = rng.standard_normal((B, 2), dtype=np.float32)
    g_scale_in = rng.standard_normal(B, dtype=np.float32)
    th = R.theta_write(s, x, y).reshape(B, 6)
    mask = stop < THRESHOLD
    thr = float(THRESHOLD)
    shd, scd = torch.tensor(np.stack([x, y], 1), device=dev), torch.tensor(s, device=dev)
    Wd, zd, sd, cd, gd, gshd, gscd = (torch.tensor(a, device=dev) for a in (W, z, stop, canvas, g, g_shift_in, g_scale_in))

    out = nan_buffer((B, cs, cs), dev)
    call(L.mog_stn_write_composite_sxy_forward, ptr(Wd), ptr(shd), ptr(scd), ptr(zd), ptr(sd), thr, ptr(cd), ptr(out), B, ws, ws,
         cs, cs, None)
    assert H.same_bits_or_nan(out.cpu().numpy(), R.write_composite(canvas, W, th, z, mask))
    inplace = cd.clone()
    call(L.mog_stn_write_composite_sxy_forward, ptr(Wd), ptr(shd), ptr(scd), ptr(zd), ptr(sd), thr, ptr(inplace), ptr(inplace), B,
         ws, ws, cs, cs, None)
    assert torch.equal(inplace, out)

    dU, d_shift, d_scale, dz = nan_buffer((B, ws, ws), dev), nan_buffer((B, 2), dev), nan_buffer((B,), dev), nan_buffer((B,), dev)
    call(L.mog_stn_write_composite_sxy_backward, ptr(Wd), ptr(shd), ptr(scd), ptr(zd), ptr(sd), thr, ptr(gd), ptr(gshd), ptr(gscd),
         ptr(dU), ptr(d_shift), ptr(d_scale), ptr(dz), B, ws, ws, cs, cs, None)
    rU, rth, _ = R.write_composite_backward(W, th, z, mask, g)
    gwin = (mask * z.astype(np.float64))[:, None, None] * g
    aU, ath = R.backward_term_magnitudes(W[..., None], th, (cs, cs), gwin[..., None])
    rz, az = dz_reference(W, th, (cs, cs), g, mask)
    r_shift, r_scale, a_shift, a_scale = sxy_chain_rule(rth, ath, s, x, y, True, g_shift_in, g_scale_in)
    dU_, dsh_, dsc_, dz_ = (t.cpu().numpy() for t in (dU, d_shift, d_scale, dz))
    assert H.grad_excess(dU_, rU, aU[..., 0]) <= 1.0
    assert H.grad_excess(dz_, rz, az) <= 1.0
    assert H.grad_excess(dsh_, r_shift, a_shift) <= 1.0
    assert H.grad_excess(dsc_, r_scale, a_scale) <= 1.0
    assert np.all(dU_[~mask] == 0) and np.all(dz_[~mask] == 0)
    assert np.array_equal(dsh_[~mask], g_shift_in[~mask]) and np.array_equal(dsc_[~mask], g_scale_in[~mask])


# ---------------------------------------------------------------------------------------------------------------------
# plain transformer(): dtheta-only mode in every class
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("src,dst", CLASSES + [
    pytest.param(256, 64, id="256to64")])   # stn_bwd_warp_kernel<false, 4>: the full-cover reads of the mix need two strips
def test_dtheta_only_mode_in_every_class(cuda_device, src, dst):
    """mog_stn_backward with dU = NULL (the AIR read site) skips the dU work -- strip passes past the first, phase 2, the
    zero fills -- and must give the same dtheta bits as the full call, which meets the fp64 oracle."""
    L = _lib.load()
    dev = cuda_device
    B = batch_size(src, dst)
    rng = np.random.default_rng(src * 1000 + dst + 3)
    th = make_thetas(B, src < dst, seed=src + dst)
    U = rng.random((B, src, src, 1), dtype=np.float32)
    g = rng.standard_normal((B, dst, dst, 1), dtype=np.float32)
    Ud, thd, gd = (torch.tensor(a, device=dev) for a in (U, th, g))
    dU, dth, dth_only = nan_buffer((B, src, src, 1), dev), nan_buffer((B, 6), dev), nan_buffer((B, 6), dev)
    call(L.mog_stn_backward, ptr(Ud), ptr(thd), ptr(gd), ptr(dU), ptr(dth), B, src, src, 1, dst, dst, 1, None)
    call(L.mog_stn_backward, ptr(Ud), ptr(thd), ptr(gd), None, ptr(dth_only), B, src, src, 1, dst, dst, 1, None)
    assert torch.equal(dth_only, dth)
    rU, rth = R.transformer_backward(U, th, (dst, dst), g)
    aU, ath = R.backward_term_magnitudes(U, th, (dst, dst), g)
    assert H.grad_excess(dU.cpu().numpy(), rU, aU) <= 1.0
    assert H.grad_excess(dth.cpu().numpy().reshape(-1, 2, 3), rth, ath) <= 1.0


# ---------------------------------------------------------------------------------------------------------------------
# batch_transformer form: u_batch_div = T, dU summed over the T transforms of a source image
# ---------------------------------------------------------------------------------------------------------------------
def batch_thetas(B, T, kind, seed):
    if kind == "general":   # every other transform general affine, the rest the mix of make_thetas
        th = make_thetas(B * T, False, seed)
        th[1::2] = [general_affine(t) for t in th[1::2]]
        return th.reshape(B, T, 6)
    s, x, y = synth.sxy_prior_like(B * T, seed=seed)
    if kind in ("full", "mixed"):
        sf, xf, yf = synth.sxy_full_cover(B * T, seed=seed + 1)
        pick = np.ones(B * T, bool) if kind == "full" else np.arange(B * T) % 2 == 1
        s, x, y = np.where(pick, sf, s), np.where(pick, xf, x), np.where(pick, yf, y)
    return R.theta_read(s, x, y).reshape(B, T, 6)


@pytest.mark.parametrize("Hs,Ho,C,T,kind", [
    # stn_bwd_warp_kernel<false, 4>, coop_zero = 1: the CTA zero-fills its group of source images in one sweep
    pytest.param(256, 64, 1, 8, "prior", id="256to64_T8_prior"),
    # same, footprint > 128 columns: two strips, accumulated over the T transforms
    pytest.param(256, 64, 1, 8, "full", id="256to64_T8_full"),
    # stn_bwd_warp_kernel<false, 4>, coop_zero = 1, two strips
    pytest.param(150, 64, 1, 3, "full", id="150to64_T3_full"),
    # stn_bwd_warp_kernel<false, 2> entering the general path for C = 3 (red.add over T), coop_zero = 0
    pytest.param(50, 28, 3, 4, "prior", id="50to28_C3_T4"),
    # stn_bwd_warp_kernel<false, 4>, coop_zero = 1, general affine: red.add on the CTA-zeroed region
    pytest.param(96, 64, 1, 4, "general", id="96to64_T4_general"),
])
def test_batch_transformer_matches_the_oracle(cuda_device, Hs, Ho, C, T, kind):
    """mog_stn_forward / mog_stn_backward with u_batch_div = T on an odd number of source images (the last CTA group has one
    warp): the forward bit-exact with the oracle's batch_transformer; dU (summed over the T transforms) and dtheta within
    tolerance of the fp64 oracle on the repeated images; the dtheta-only call gives the same dtheta bits."""
    L = _lib.load()
    dev = cuda_device
    B = 5
    rng = np.random.default_rng(Hs * 100 + Ho + C + T)
    U = rng.random((B, Hs, Hs, C), dtype=np.float32)
    th = batch_thetas(B, T, kind, seed=Hs + T)
    g = rng.standard_normal((B * T, Ho, Ho, C), dtype=np.float32)
    Ud, thd, gd = (torch.tensor(a, device=dev) for a in (U, th, g))
    out = nan_buffer((B * T, Ho, Ho, C), dev)
    call(L.mog_stn_forward, ptr(Ud), ptr(thd), ptr(out), B * T, Hs, Hs, C, Ho, Ho, T, None)
    assert H.same_bits_or_nan(out.cpu().numpy(), R.batch_transformer(U, th, (Ho, Ho)))

    dU, dth, dth_only = nan_buffer((B, Hs, Hs, C), dev), nan_buffer((B * T, 6), dev), nan_buffer((B * T, 6), dev)
    call(L.mog_stn_backward, ptr(Ud), ptr(thd), ptr(gd), ptr(dU), ptr(dth), B * T, Hs, Hs, C, Ho, Ho, T, None)
    call(L.mog_stn_backward, ptr(Ud), ptr(thd), ptr(gd), None, ptr(dth_only), B * T, Hs, Hs, C, Ho, Ho, T, None)
    Urep, th2 = np.repeat(U, T, axis=0), th.reshape(B * T, 6)
    rU, rth = R.transformer_backward(Urep, th2, (Ho, Ho), g)
    aU, ath = R.backward_term_magnitudes(Urep, th2, (Ho, Ho), g)
    rU, aU = rU.reshape(B, T, Hs, Hs, C).sum(1), aU.reshape(B, T, Hs, Hs, C).sum(1)
    assert H.grad_excess(dU.cpu().numpy(), rU, aU) <= 1.0
    assert H.grad_excess(dth.cpu().numpy().reshape(-1, 2, 3), rth, ath) <= 1.0
    assert torch.equal(dth_only, dth)


def test_batch_host_entry_point_matches_the_device_call_at_256(cuda_device):
    """HostSampler.batch_fwd_bwd (mog_stn_batch_fwd_bwd_host, the end-to-end read leg of bench.py) at 256 x 256 -> 64 x 64,
    T = 8, with a ragged last chunk of one source image: the same bits as the device call with u_batch_div = T."""
    from mog_asr_b200.host_api import HostSampler
    L = _lib.load()
    dev = cuda_device
    B, T, Hs, Ho = 5, 8, 256, 64
    rng = np.random.default_rng(256)
    U = rng.random((B, Hs, Hs, 1), dtype=np.float32)
    th = batch_thetas(B, T, "mixed", seed=31)
    g = rng.standard_normal((B, T, Ho, Ho, 1), dtype=np.float32)
    Ud, thd, gd = (torch.tensor(a, device=dev) for a in (U, th, g))
    out, dU, dth = nan_buffer((B * T, Ho, Ho, 1), dev), nan_buffer((B, Hs, Hs, 1), dev), nan_buffer((B * T, 6), dev)
    call(L.mog_stn_forward, ptr(Ud), ptr(thd), ptr(out), B * T, Hs, Hs, 1, Ho, Ho, T, None)
    call(L.mog_stn_backward, ptr(Ud), ptr(thd), ptr(gd), ptr(dU), ptr(dth), B * T, Hs, Hs, 1, Ho, Ho, T, None)
    hs = HostSampler(dev, (Hs, Hs), (Ho, Ho), 1, chunk=2, nstreams=2, transforms=T)
    pin = [torch.from_numpy(a).pin_memory() for a in (U, th, g)]
    h_out, h_dU, h_dth = hs.batch_fwd_bwd(*pin)
    assert torch.equal(h_out, out.cpu()) and torch.equal(h_dU, dU.cpu()) and torch.equal(h_dth.reshape(-1, 6), dth.cpu())
