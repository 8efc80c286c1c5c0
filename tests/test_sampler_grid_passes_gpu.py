"""GPU parity of the sampler's other forms -- the fused write + composite, the (s, x, y) entry points, the batched
(``u_batch_div > 1``) forward and backward and the corner probe -- past one grid pass.

Every sampler kernel walks its images in a group-stride loop: a CTA of kWarpsPerCta = 2 warps takes 2 images per iteration
and ``grid_for`` caps the grid at ``sm_count() * ctas_per_sm`` (csrc/mog_stn.cu).  The forward and the streaming backward
cap at 32 CTAs per SM, the source-column backward at what the occupancy query allows (at most 32), and the corner probe runs
one 256-thread CTA per image with 8 CTAs per SM.  So ``B = 64 * n_sm + 3`` images (``16 * n_sm + 1`` for the corner probe)
take more than one pass of every one of these kernels, whatever the occupancy query returns, and the odd B leaves the last
CTA group with a single warp.  Every image is distinct (its own U, gradients, z_pres, stop_sum and add-ins; theta kinds
cycle with period 9), so a kernel that reads another image's data on a later pass gives different values.

Two references:
  1. the same entry point called on consecutive slices of at most ``2 * n_sm`` images, each of which fits in one pass at
     any occupancy (n_sm CTAs or fewer), compared on every image: bit-equal wherever the kernel has no atomics (forwards,
     dtheta, dz, d_shift / d_scale, the dU of separable thetas); the dU of a general-affine theta (summed by red.add, in no
     fixed order) within twice ``GRAD_RTOL`` of each entry's sum of |terms|, since each call is within ``GRAD_RTOL`` of the
     exact sum;
  2. the fp64 oracle on a sample of about 60 images -- the first and last four, every image from ``64 * n_sm - 2`` on (the
     start of the forward's second pass) and a stride through the rest: forwards and corners bit-exact, gradients within
     ``GRAD_RTOL`` of the sum of |terms| entering each entry (DESIGN.md section 4).
Every output buffer is pre-filled with NaN through the C ABI (the corner planes with INT32_MIN) and must come back finite."""
import time

import numpy as np
import pytest
import torch

from mog_asr_b200 import _lib
from oracle import stn_ref_c as RC
from oracle import stn_ref_numpy as R
from tests import helpers as H
from tests.test_sampler_paths_gpu import (CLASSES, KINDS, STOP_SUM, THRESHOLD, Z_PRES, call, dz_reference, make_thetas,
                                          nan_buffer, separable, sxy_chain_rule, sxy_inputs)

pytestmark = pytest.mark.gpu

POISON_I32 = -(2 ** 31)


def grid_pass_batch(dev, per_sm=64, extra=3):
    """(n_sm, B) with B = per_sm * n_sm + extra: past one grid pass of every sampler kernel (per_sm = 64: 32 CTAs of 2
    warps per SM, the largest cap any of them can get; the corner probe: 16, 8 CTAs of one image each, times two)."""
    n = torch.cuda.get_device_properties(dev).multi_processor_count
    B = per_sm * n + extra
    print(f"B = {B}, one grid pass at most {per_sm * n} images ({n} SMs)")
    assert B > per_sm * n
    return n, B


def one_pass_slices(B, n, per=1):
    """[lo, hi) slices of at most 2 * n_sm images (per = transforms per image): n_sm CTAs or fewer, one pass at any cap."""
    step = max(1, (2 * n) // per)
    return [(lo, min(B, lo + step)) for lo in range(0, B, step)]


def sample_indices(B, n, per_sm=64):
    """the first and last four images, every image from per_sm * n_sm - 2 on and a stride through the rest: about 60"""
    idx = set(range(4)) | set(range(B - 4, B)) | set(range(per_sm * n - 2, B)) | set(range(4, B - 4, max(1, B // 48)))
    return np.array(sorted(idx))


def at(t, lo):
    """device pointer to image lo of t (None stays None)"""
    return t[lo:].data_ptr() if t is not None else None


def run_sliced(fn, B, n, per=1):
    """fn(lo, nb) on each one-pass slice"""
    for lo, hi in one_pass_slices(B, n, per):
        fn(lo, hi - lo)


def run_whole_and_sliced(fns, B, n, per=1):
    """fns[0](0, B) on the whole batch, then fns[1](lo, nb) on one-pass slices: the reference buffers"""
    fns[0](0, B)
    run_sliced(fns[1], B, n, per)


def same_bits(a, b):
    return torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


def finite(*ts):
    return all(bool(torch.isfinite(t).all()) for t in ts)


def within_sum_of_terms(a, b, mag):
    """|a - b| <= 2 GRAD_RTOL * mag per entry: a and b are each within GRAD_RTOL * mag of the exact sum"""
    return bool(((a - b).abs() <= 2 * H.GRAD_RTOL * mag).all())


def cpu(t, idx):
    return t[torch.as_tensor(idx, device=t.device)].cpu().numpy()


def elapsed(t0):
    print(f"wall time {time.perf_counter() - t0:.1f} s")


# ---------------------------------------------------------------------------------------------------------------------
# fused write + composite, theta given
# ---------------------------------------------------------------------------------------------------------------------
def composite_batch(B, ws, cs, seed, dev):
    """window, theta, z_pres, stop_sum, canvas, gcanvas on the device: every image its own draws.  z_pres in (0, 1), exactly 0
    or negative and stop_sum below, exactly at or above the threshold, paired with the theta kinds as in
    test_sampler_paths_gpu.composite_inputs.  Canvases hold no -0.0 (the in-place form skips canvas + 0)."""
    gen = torch.Generator(device=dev).manual_seed(seed)
    W = torch.rand((B, ws, ws), device=dev, generator=gen)
    canvas = torch.rand((B, cs, cs), device=dev, generator=gen) * 0.99 + 0.01
    g = torch.randn((B, cs, cs), device=dev, generator=gen)
    rng = np.random.default_rng(seed)
    th = make_thetas(B, True, seed)
    z = rng.uniform(0.05, 0.95, B).astype(np.float32)
    stop = rng.uniform(0.0, 0.85, B).astype(np.float32)
    for b in range(B):
        k = (b + 4 * (b // len(KINDS))) % len(KINDS)
        if Z_PRES[k] is not None:
            z[b] = -z[b] if Z_PRES[k] < 0 else Z_PRES[k]
        if STOP_SUM[k] == THRESHOLD:
            stop[b] = THRESHOLD
        elif STOP_SUM[k] > THRESHOLD:
            stop[b] += 1.0
    return W, th, z, stop, canvas, g


@pytest.mark.parametrize("ws,cs", CLASSES)
def test_write_composite_past_one_grid_pass(cuda_device, ws, cs):
    """mog_stn_write_composite_forward / _backward on B = 64 n_sm + 3 images: out of place and in place bit-equal to
    one-pass slices and to each other, inactive images untouched in place; the backward (full, dU-less) equal to one-pass
    slices on every image, run-to-run deterministic, and within tolerance of the fp64 oracle on the sample."""
    t0 = time.perf_counter()
    L = _lib.load()
    dev = cuda_device
    n, B = grid_pass_batch(dev)
    W, th, z, stop, canvas, g = composite_batch(B, ws, cs, ws * 1000 + cs + 11, dev)
    mask = stop < THRESHOLD
    thd, zd, sd = (torch.tensor(a, device=dev) for a in (th, z, stop))
    thr = float(THRESHOLD)

    def fwd(cin, cout):
        return lambda lo, nb: call(L.mog_stn_write_composite_forward, at(W, lo), at(thd, lo), at(zd, lo), at(sd, lo), thr,
                                   at(cin, lo), at(cout, lo), nb, ws, ws, cs, cs, None)

    out, out1 = nan_buffer((B, cs, cs), dev), nan_buffer((B, cs, cs), dev)
    run_whole_and_sliced((fwd(canvas, out), fwd(canvas, out1)), B, n)
    inplace, inplace1 = canvas.clone(), canvas.clone()
    run_whole_and_sliced((fwd(inplace, inplace), fwd(inplace1, inplace1)), B, n)
    assert finite(out, inplace)
    assert same_bits(out, out1) and same_bits(inplace, inplace1) and same_bits(inplace, out)
    inactive = torch.tensor(~mask, device=dev)
    assert same_bits(inplace[inactive], canvas[inactive])

    def grads(want_dU=True):
        return [nan_buffer((B, ws, ws), dev) if want_dU else None, nan_buffer((B, 6), dev), nan_buffer((B,), dev)]

    def bwd(bufs, gc=g, zp=zd):
        dU, dth, dz = bufs
        return lambda lo, nb: call(L.mog_stn_write_composite_backward, at(W, lo), at(thd, lo), at(zp, lo), at(sd, lo), thr,
                                   at(gc, lo), at(dU, lo), at(dth, lo), at(dz, lo), nb, ws, ws, cs, cs, None)

    full, full1, again, nodU, nodU1 = grads(), grads(), grads(), grads(False), grads(False)
    run_whole_and_sliced((bwd(full), bwd(full1)), B, n)
    run_whole_and_sliced((bwd(nodU), bwd(nodU1)), B, n)
    bwd(again)(0, B)
    dU, dth, dz = full
    assert finite(*full)
    sep = torch.tensor(separable(th), device=dev)
    aff = ~sep
    for x, x1, x2 in zip(full[1:], full1[1:], again[1:]):   # dtheta and dz: warp sums, no atomics, every image
        assert same_bits(x, x1) and same_bits(x, x2)
    assert same_bits(nodU[1], dth) and same_bits(nodU[2], dz) and same_bits(nodU1[1], dth) and same_bits(nodU1[2], dz)
    assert same_bits(dU[sep], full1[0][sep]) and same_bits(dU[sep], again[0][sep])
    # general affine: Sigma|terms| of each dU entry is the same backward on |g| and |z| (every in-range weight is >= 0)
    mag = grads()
    run_sliced(bwd(mag, g.abs(), zd.abs()), B, n)
    assert within_sum_of_terms(dU[aff], full1[0][aff], mag[0][aff])
    assert within_sum_of_terms(dU[aff], again[0][aff], mag[0][aff])
    assert bool((dU[inactive] == 0).all() and (dth[inactive] == 0).all() and (dz[inactive] == 0).all())

    idx = sample_indices(B, n)
    Ws, ths, zs, ms, cvs, gs = cpu(W, idx), th[idx], z[idx], mask[idx], cpu(canvas, idx), cpu(g, idx)
    assert np.array_equal(cpu(out, idx).view(np.uint32), R.write_composite(cvs, Ws, ths, zs, ms).view(np.uint32))
    rU, rth, _ = R.write_composite_backward(Ws, ths, zs, ms, gs)
    gwin = (ms * zs.astype(np.float64))[:, None, None] * gs
    aU, ath = R.backward_term_magnitudes(Ws[..., None], ths, (cs, cs), gwin[..., None])
    rz, az = dz_reference(Ws, ths, (cs, cs), gs, ms)
    assert H.grad_excess(cpu(dU, idx), rU, aU[..., 0]) <= 1.0
    assert H.grad_excess(cpu(dth, idx).reshape(-1, 2, 3), rth, ath) <= 1.0
    assert H.grad_excess(cpu(dz, idx), rz, az) <= 1.0
    elapsed(t0)


# ---------------------------------------------------------------------------------------------------------------------
# (s, x, y) entry points
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("src,dst", CLASSES)
def test_read_sxy_past_one_grid_pass(cuda_device, src, dst):
    """mog_stn_read_sxy_forward / _backward on B = 64 n_sm + 3 images, with and without dU and with non-zero d_shift /
    d_scale add-ins: every output bit-equal to one-pass slices and run to run; the dU-less call gives the same d_shift /
    d_scale; the glimpse bit-exact and the gradients within tolerance of the fp64 oracle on the sample."""
    t0 = time.perf_counter()
    L = _lib.load()
    dev = cuda_device
    n, B = grid_pass_batch(dev)
    gen = torch.Generator(device=dev).manual_seed(src * 1000 + dst + 17)
    U = torch.rand((B, src, src), device=dev, generator=gen)
    g = torch.randn((B, dst, dst), device=dev, generator=gen)
    gsh = torch.randn((B, 2), device=dev, generator=gen)
    gsc = torch.randn((B,), device=dev, generator=gen)
    s, x, y = sxy_inputs(B, seed=src + dst + 5)
    shd, scd = torch.tensor(np.stack([x, y], 1), device=dev), torch.tensor(s, device=dev)

    def fwd(o):
        return lambda lo, nb: call(L.mog_stn_read_sxy_forward, at(U, lo), at(shd, lo), at(scd, lo), at(o, lo), nb, src, src, dst,
                                   dst, None)

    out, out1 = nan_buffer((B, dst, dst), dev), nan_buffer((B, dst, dst), dev)
    run_whole_and_sliced((fwd(out), fwd(out1)), B, n)
    assert finite(out) and same_bits(out, out1)

    def grads(want_dU=True):
        return [nan_buffer((B, src, src), dev) if want_dU else None, nan_buffer((B, 2), dev), nan_buffer((B,), dev)]

    def bwd(bufs):
        dU, d_shift, d_scale = bufs
        return lambda lo, nb: call(L.mog_stn_read_sxy_backward, at(U, lo), at(shd, lo), at(scd, lo), at(g, lo), at(gsh, lo),
                                   at(gsc, lo), at(dU, lo), at(d_shift, lo), at(d_scale, lo), nb, src, src, dst, dst, None)

    full, full1, again, nodU, nodU1 = grads(), grads(), grads(), grads(False), grads(False)
    run_whole_and_sliced((bwd(full), bwd(full1)), B, n)
    run_whole_and_sliced((bwd(nodU), bwd(nodU1)), B, n)
    bwd(again)(0, B)
    assert finite(*full)
    for k in range(3):
        assert same_bits(full[k], full1[k]) and same_bits(full[k], again[k])
    for k in (1, 2):
        assert same_bits(nodU[k], full[k]) and same_bits(nodU1[k], full[k])

    idx = sample_indices(B, n)
    Us, gs = cpu(U, idx)[..., None], cpu(g, idx)[..., None]
    th = R.theta_read(s[idx], x[idx], y[idx]).reshape(-1, 6)
    assert np.array_equal(cpu(out, idx).view(np.uint32), R.transformer(Us, th, (dst, dst))[..., 0].view(np.uint32))
    rU, rth = R.transformer_backward(Us, th, (dst, dst), gs)
    aU, ath = R.backward_term_magnitudes(Us, th, (dst, dst), gs)
    r_shift, r_scale, a_shift, a_scale = sxy_chain_rule(rth, ath, s[idx], x[idx], y[idx], False, cpu(gsh, idx), cpu(gsc, idx))
    assert H.grad_excess(cpu(full[0], idx), rU[..., 0], aU[..., 0]) <= 1.0
    assert H.grad_excess(cpu(full[1], idx), r_shift, a_shift) <= 1.0
    assert H.grad_excess(cpu(full[2], idx), r_scale, a_scale) <= 1.0
    elapsed(t0)


@pytest.mark.parametrize("ws,cs", CLASSES)
def test_write_composite_sxy_past_one_grid_pass(cuda_device, ws, cs):
    """mog_stn_write_composite_sxy_forward / _backward on B = 64 n_sm + 3 images: the canvas out of place and in place, dU,
    dz, d_shift and d_scale (with add-ins) bit-equal to one-pass slices and run to run; inactive images get exactly the
    add-ins and zero dU / dz; canvas bit-exact and gradients within tolerance of the fp64 oracle on the sample."""
    t0 = time.perf_counter()
    L = _lib.load()
    dev = cuda_device
    n, B = grid_pass_batch(dev)
    W, _, z, stop, canvas, g = composite_batch(B, ws, cs, ws * 1000 + cs + 12, dev)
    gen = torch.Generator(device=dev).manual_seed(ws + cs + 13)
    gsh = torch.randn((B, 2), device=dev, generator=gen)
    gsc = torch.randn((B,), device=dev, generator=gen)
    s, x, y = sxy_inputs(B, seed=ws * 3 + cs + 1)
    mask = stop < THRESHOLD
    thr = float(THRESHOLD)
    shd, scd, zd, sd = (torch.tensor(a, device=dev) for a in (np.stack([x, y], 1), s, z, stop))

    def fwd(cin, cout):
        return lambda lo, nb: call(L.mog_stn_write_composite_sxy_forward, at(W, lo), at(shd, lo), at(scd, lo), at(zd, lo),
                                   at(sd, lo), thr, at(cin, lo), at(cout, lo), nb, ws, ws, cs, cs, None)

    out, out1 = nan_buffer((B, cs, cs), dev), nan_buffer((B, cs, cs), dev)
    run_whole_and_sliced((fwd(canvas, out), fwd(canvas, out1)), B, n)
    inplace, inplace1 = canvas.clone(), canvas.clone()
    run_whole_and_sliced((fwd(inplace, inplace), fwd(inplace1, inplace1)), B, n)
    assert finite(out, inplace)
    assert same_bits(out, out1) and same_bits(inplace, inplace1) and same_bits(inplace, out)
    inactive = torch.tensor(~mask, device=dev)
    assert same_bits(inplace[inactive], canvas[inactive])

    def grads():
        return [nan_buffer((B, ws, ws), dev), nan_buffer((B, 2), dev), nan_buffer((B,), dev), nan_buffer((B,), dev)]

    def bwd(bufs):
        dU, d_shift, d_scale, dz = bufs
        return lambda lo, nb: call(L.mog_stn_write_composite_sxy_backward, at(W, lo), at(shd, lo), at(scd, lo), at(zd, lo),
                                   at(sd, lo), thr, at(g, lo), at(gsh, lo), at(gsc, lo), at(dU, lo), at(d_shift, lo),
                                   at(d_scale, lo), at(dz, lo), nb, ws, ws, cs, cs, None)

    full, full1, again = grads(), grads(), grads()
    run_whole_and_sliced((bwd(full), bwd(full1)), B, n)
    bwd(again)(0, B)
    dU, d_shift, d_scale, dz = full
    assert finite(*full)
    for k in range(4):
        assert same_bits(full[k], full1[k]) and same_bits(full[k], again[k])
    assert bool((dU[inactive] == 0).all() and (dz[inactive] == 0).all())
    assert same_bits(d_shift[inactive], gsh[inactive]) and same_bits(d_scale[inactive], gsc[inactive])

    idx = sample_indices(B, n)
    Ws, zs, ms, cvs, gs = cpu(W, idx), z[idx], mask[idx], cpu(canvas, idx), cpu(g, idx)
    th = R.theta_write(s[idx], x[idx], y[idx]).reshape(-1, 6)
    assert np.array_equal(cpu(out, idx).view(np.uint32), R.write_composite(cvs, Ws, th, zs, ms).view(np.uint32))
    rU, rth, _ = R.write_composite_backward(Ws, th, zs, ms, gs)
    gwin = (ms * zs.astype(np.float64))[:, None, None] * gs
    aU, ath = R.backward_term_magnitudes(Ws[..., None], th, (cs, cs), gwin[..., None])
    rz, az = dz_reference(Ws, th, (cs, cs), gs, ms)
    r_shift, r_scale, a_shift, a_scale = sxy_chain_rule(rth, ath, s[idx], x[idx], y[idx], True, cpu(gsh, idx), cpu(gsc, idx))
    assert H.grad_excess(cpu(dU, idx), rU, aU[..., 0]) <= 1.0
    assert H.grad_excess(cpu(dz, idx), rz, az) <= 1.0
    assert H.grad_excess(cpu(d_shift, idx), r_shift, a_shift) <= 1.0
    assert H.grad_excess(cpu(d_scale, idx), r_scale, a_scale) <= 1.0
    elapsed(t0)


# ---------------------------------------------------------------------------------------------------------------------
# batch_transformer form: u_batch_div = T, dU summed over the T transforms of a source image
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("Hs,Ho,T", [
    pytest.param(50, 28, 4, id="50to28_T4"),   # stn_bwd_warp_kernel<false, 2>, coop_zero = 0: each warp zero-fills its image
    pytest.param(96, 64, 2, id="96to64_T2"),   # stn_bwd_warp_kernel<false, 4>, coop_zero = 1: the CTA sweeps its group
])
def test_batch_transformer_past_one_grid_pass(cuda_device, Hs, Ho, T):
    """mog_stn_forward / mog_stn_backward with u_batch_div = T on Bsrc = 64 n_sm + 3 source images, the theta kinds of
    make_thetas mixed over the transforms (general affine ones included): the forward, dtheta, the dtheta-only call and the
    dU of source images without a general-affine transform bit-equal to one-pass slices and run to run, the other dU within
    the sum of |terms|; the forward bit-exact and the gradients within tolerance of the fp64 oracle on the sample."""
    t0 = time.perf_counter()
    L = _lib.load()
    dev = cuda_device
    n, B = grid_pass_batch(dev)
    gen = torch.Generator(device=dev).manual_seed(Hs * 100 + Ho + T)
    U = torch.rand((B, Hs, Hs, 1), device=dev, generator=gen)
    g = torch.randn((B * T, Ho, Ho, 1), device=dev, generator=gen)
    th = make_thetas(B * T, False, seed=Hs + Ho + T)
    thd = torch.tensor(th, device=dev)

    def fwd(o):
        return lambda lo, nb: call(L.mog_stn_forward, at(U, lo), at(thd, lo * T), at(o, lo * T), nb * T, Hs, Hs, 1, Ho, Ho, T,
                                   None)

    out, out1 = nan_buffer((B * T, Ho, Ho, 1), dev), nan_buffer((B * T, Ho, Ho, 1), dev)
    run_whole_and_sliced((fwd(out), fwd(out1)), B, n, per=T)
    assert finite(out) and same_bits(out, out1)

    def grads(want_dU=True):
        return [nan_buffer((B, Hs, Hs, 1), dev) if want_dU else None, nan_buffer((B * T, 6), dev)]

    def bwd(bufs, go=g):
        dU, dth = bufs
        return lambda lo, nb: call(L.mog_stn_backward, at(U, lo), at(thd, lo * T), at(go, lo * T), at(dU, lo), at(dth, lo * T),
                                   nb * T, Hs, Hs, 1, Ho, Ho, T, None)

    full, full1, again, nodU, nodU1 = grads(), grads(), grads(), grads(False), grads(False)
    run_whole_and_sliced((bwd(full), bwd(full1)), B, n, per=T)
    run_whole_and_sliced((bwd(nodU), bwd(nodU1)), B, n, per=T)
    bwd(again)(0, B)
    dU, dth = full
    assert finite(dU, dth)
    assert same_bits(dth, full1[1]) and same_bits(dth, again[1]) and same_bits(nodU[1], dth) and same_bits(nodU1[1], dth)
    sep_src = torch.tensor(separable(th).reshape(B, T).all(1), device=dev)
    assert same_bits(dU[sep_src], full1[0][sep_src]) and same_bits(dU[sep_src], again[0][sep_src])
    mag = grads()
    run_sliced(bwd(mag, g.abs()), B, n, per=T)
    assert within_sum_of_terms(dU[~sep_src], full1[0][~sep_src], mag[0][~sep_src])
    assert within_sum_of_terms(dU[~sep_src], again[0][~sep_src], mag[0][~sep_src])

    idx = sample_indices(B, n)
    tidx = (idx[:, None] * T + np.arange(T)).reshape(-1)
    Us, ths, gs = cpu(U, idx), th[tidx], cpu(g, tidx)
    assert np.array_equal(cpu(out, tidx).view(np.uint32), R.batch_transformer(Us, ths.reshape(-1, T, 6), (Ho, Ho)).view(np.uint32))
    Urep = np.repeat(Us, T, axis=0)
    rU, rth = R.transformer_backward(Urep, ths, (Ho, Ho), gs)
    aU, ath = R.backward_term_magnitudes(Urep, ths, (Ho, Ho), gs)
    rU, aU = rU.reshape(-1, T, Hs, Hs, 1).sum(1), aU.reshape(-1, T, Hs, Hs, 1).sum(1)
    assert H.grad_excess(cpu(dU, idx), rU, aU) <= 1.0
    assert H.grad_excess(cpu(dth, tidx).reshape(-1, 2, 3), rth, ath) <= 1.0
    elapsed(t0)


# ---------------------------------------------------------------------------------------------------------------------
# corner probe: one CTA per image, 8 per SM
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("Hs,Ho,write", [pytest.param(50, 28, False, id="read_50to28"),
                                         pytest.param(28, 50, True, id="write_28to50")])
def test_corners_past_one_grid_pass(cuda_device, Hs, Ho, write):
    """mog_stn_corners on B = 16 n_sm + 1 images, separable and general-affine thetas mixed: bit-equal to one-pass slices
    on every image and bit-exact with the C oracle's corners on the sample."""
    t0 = time.perf_counter()
    L = _lib.load()
    dev = cuda_device
    n, B = grid_pass_batch(dev, per_sm=16, extra=1)
    N = Ho * Ho
    th = make_thetas(B, write, seed=Hs + Ho + 21)
    thd = torch.tensor(th, device=dev)
    corners = torch.full((4, B, N), POISON_I32, dtype=torch.int32, device=dev)
    call(L.mog_stn_corners, thd.data_ptr(), corners.data_ptr(), B, Hs, Hs, Ho, Ho, None)
    sliced = torch.full((4, B, N), POISON_I32, dtype=torch.int32, device=dev)
    for lo, hi in one_pass_slices(B, n):   # the four planes of a call are [nb][N] each: copy the slice's planes in
        part = torch.full((4, hi - lo, N), POISON_I32, dtype=torch.int32, device=dev)
        call(L.mog_stn_corners, at(thd, lo), part.data_ptr(), hi - lo, Hs, Hs, Ho, Ho, None)
        sliced[:, lo:hi] = part
    assert bool((corners >= 0).all() and (corners < Hs).all())
    assert torch.equal(corners, sliced)
    idx = sample_indices(B, n, per_sm=16)
    _, ref = RC.forward(np.zeros((len(idx), Hs, Hs, 1), np.float32), th[idx], (Ho, Ho), want_corners=True)
    assert np.array_equal(corners[:, torch.as_tensor(idx, device=dev)].cpu().numpy(), ref)
    elapsed(t0)
