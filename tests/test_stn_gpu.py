"""GPU parity tests of the sampler: CUDA path (through the C ABI) vs the oracle.

Contract: corner indices bit-exact; forward values bit-exact for finite inputs (same operation order,
no FMA) with the SURVEY A.1 bound as the documented tolerance; gradients within GRAD_RTOL of the fp64
oracle relative to the sum of |terms| (atomic / tree order makes them non-bit-exact)."""
import numpy as np
import pytest
import torch

import mog_asr_b200 as M
from mog_asr_b200 import _lib, synth
from oracle import stn_ref_numpy as R
from oracle import stn_ref_c as RC
from tests import helpers as H

pytestmark = pytest.mark.gpu


def run_fwd_bwd(dev, U, theta, out_size, gout, need_dU=True):
    Ut = torch.tensor(U, device=dev, requires_grad=need_dU)
    tt = torch.tensor(theta, device=dev, requires_grad=True)
    out = M.transformer(Ut, tt, tuple(int(v) for v in out_size))
    out.backward(torch.tensor(gout, device=dev))
    torch.cuda.synchronize()
    return (out.detach().cpu().numpy(), Ut.grad.cpu().numpy() if need_dU else None,
            tt.grad.cpu().numpy().reshape(-1, 2, 3))


@pytest.mark.parametrize("name", H.STN_CASES)
def test_golden_forward_corners_backward(cuda_device, name):
    d = H.load(name)
    Hs, Ws = d["U"].shape[1:3]
    corners = M.stn_corners(torch.tensor(d["theta"], device=cuda_device), (Hs, Ws), d["out_size"]).cpu().numpy()
    assert np.array_equal(corners, d["corners"].reshape(corners.shape)), "corner indices must be bit-exact"
    out, dU, dth = run_fwd_bwd(cuda_device, d["U"], d["theta"], d["out_size"], d["gout"])
    # stated tolerance (always checked) ...
    B, C = out.shape[0], d["U"].shape[-1]
    bound = H.FWD_EPS_FACTOR * H.EPS32 * d["wsum"].reshape(B, -1, 1) * np.abs(d["U"]).max()
    err = np.abs(out - d["out"]).reshape(B, -1, C)
    fin = np.isfinite(d["out"]).reshape(B, -1, C)
    assert np.all((err <= bound) | ~fin)
    # ... and the stronger property the kernels are written for
    assert H.same_bits_or_nan(out, d["out"]), "forward is expected to be bit-exact with the oracle"
    assert H.grad_excess(dU, d["dU"], d["absdU"]) <= 1.0
    assert H.grad_excess(dth, d["dtheta"], d["absdtheta"]) <= 1.0


def test_dtheta_only_mode_matches_full_mode(cuda_device):
    d = H.load("read_50_28")
    _, _, dth_full = run_fwd_bwd(cuda_device, d["U"], d["theta"], d["out_size"], d["gout"], need_dU=True)
    _, dU, dth_only = run_fwd_bwd(cuda_device, d["U"], d["theta"], d["out_size"], d["gout"], need_dU=False)
    assert dU is None
    assert np.array_equal(dth_full, dth_only)


@pytest.mark.parametrize("Hs,Ho,direction", [(50, 28, "read"), (50, 28, "write"), (64, 28, "read"),
                                              (64, 28, "write"), (128, 64, "read"), (256, 64, "read"),
                                              (256, 64, "write"), (256, 28, "read")])
@pytest.mark.parametrize("regime", ["prior", "full"])
def test_seeded_parity_vs_c_oracle(cuda_device, Hs, Ho, direction, regime):
    """Config-5 shapes at a batch the oracle finishes in seconds."""
    B = 48 if Hs <= 64 else 12
    rng = np.random.default_rng(Hs * 1000 + Ho)
    s, x, y = (synth.sxy_prior_like if regime == "prior" else synth.sxy_full_cover)(B, seed=11)
    if direction == "read":
        U = rng.random((B, Hs, Hs, 1), dtype=np.float32)
        th, out_size = synth.theta_read(s, x, y), (Ho, Ho)
    else:
        U = rng.random((B, Ho, Ho, 1), dtype=np.float32)
        th, out_size = synth.theta_write(s, x, y), (Hs, Hs)
    g = rng.normal(size=(B, out_size[0], out_size[1], 1)).astype(np.float32)
    ref_out, ref_c = RC.forward(U, th, out_size, want_corners=True)
    corners = M.stn_corners(torch.tensor(th, device=cuda_device), U.shape[1:3], out_size).cpu().numpy()
    assert np.array_equal(corners, ref_c)
    out, dU, dth = run_fwd_bwd(cuda_device, U, th, out_size, g)
    assert H.same_bits_or_nan(out, ref_out)
    dU64, dth64 = R.transformer_backward(U, th, out_size, g, dtype=np.float64)
    aU, ath = R.backward_term_magnitudes(U, th, out_size, g)
    assert H.grad_excess(dU, dU64, aU) <= 1.0
    assert H.grad_excess(dth, dth64, ath) <= 1.0


def test_general_affine_and_channels(cuda_device):
    rng = np.random.default_rng(21)
    B, Hs, Ws, C, Ho, Wo = 20, 37, 41, 4, 19, 23
    U = rng.normal(size=(B, Hs, Ws, C)).astype(np.float32)
    th = (np.tile(np.asarray([[0.8, 0, 0, 0, 0.8, 0]], np.float32), (B, 1)) + rng.normal(0, 0.3, (B, 6))).astype(np.float32)
    g = rng.normal(size=(B, Ho, Wo, C)).astype(np.float32)
    ref_out, ref_c = RC.forward(U, th, (Ho, Wo), want_corners=True)
    assert np.array_equal(M.stn_corners(torch.tensor(th, device=cuda_device), (Hs, Ws), (Ho, Wo)).cpu().numpy(), ref_c)
    out, dU, dth = run_fwd_bwd(cuda_device, U, th, (Ho, Wo), g)
    assert H.same_bits_or_nan(out, ref_out)
    dU64, dth64 = R.transformer_backward(U, th, (Ho, Wo), g, dtype=np.float64)
    aU, ath = R.backward_term_magnitudes(U, th, (Ho, Wo), g)
    assert H.grad_excess(dU, dU64, aU) <= 1.0
    assert H.grad_excess(dth, dth64, ath) <= 1.0


def test_batch_transformer_matches_repeat(cuda_device):
    rng = np.random.default_rng(22)
    B, T = 6, 8
    U = rng.random((B, 50, 50, 1), dtype=np.float32)
    s, x, y = synth.sxy_prior_like(B * T, seed=5)
    th = synth.theta_read(s, x, y).reshape(B, T, 6)
    g = rng.normal(size=(B * T, 28, 28, 1)).astype(np.float32)
    Ut = torch.tensor(U, device=cuda_device, requires_grad=True)
    tt = torch.tensor(th, device=cuda_device, requires_grad=True)
    out = M.batch_transformer(Ut, tt, (28, 28))
    assert out.shape == (B * T, 28, 28, 1)
    out.backward(torch.tensor(g, device=cuda_device))
    ref = R.batch_transformer(U, th, (28, 28))
    assert H.same_bits_or_nan(out.detach().cpu().numpy(), ref)
    Urep = np.repeat(U, T, axis=0)
    dU64, dth64 = R.transformer_backward(Urep, th.reshape(-1, 6), (28, 28), g)
    aU, ath = R.backward_term_magnitudes(Urep, th.reshape(-1, 6), (28, 28), g)
    dU64 = dU64.reshape(B, T, 50, 50, 1).sum(1)
    aU = aU.reshape(B, T, 50, 50, 1).sum(1)
    assert H.grad_excess(Ut.grad.cpu().numpy(), dU64, aU) <= 1.0
    assert H.grad_excess(tt.grad.cpu().numpy().reshape(-1, 2, 3), dth64, ath) <= 1.0


def test_empty_and_ragged_inputs(cuda_device):
    out = M.transformer(torch.zeros((0, 50, 50, 1), device=cuda_device), torch.zeros((0, 6), device=cuda_device), (28, 28))
    assert out.shape == (0, 28, 28, 1)
    # theta as [B,2,3], non-contiguous U, float64 inputs: cast/reshaped like transformer.py:101,144-145
    rng = np.random.default_rng(3)
    U = rng.random((5, 13, 50, 2))
    th = rng.normal(0, 0.5, (5, 2, 3))
    Ut = torch.tensor(U, device=cuda_device).transpose(1, 2)          # [5,50,13,2] view
    out = M.transformer(Ut, torch.tensor(th, device=cuda_device), (7, 9))
    ref = R.transformer(np.ascontiguousarray(U.transpose(0, 2, 1, 3)).astype(np.float32), th.astype(np.float32), (7, 9))
    assert H.same_bits_or_nan(out.cpu().numpy(), ref)
    with pytest.raises(ValueError):
        M.transformer(torch.zeros((2, 5, 5, 1), device=cuda_device), torch.zeros((3, 6), device=cuda_device), (2, 2))


def test_nan_theta_propagates_and_stays_in_bounds(cuda_device):
    U = torch.ones((2, 9, 9, 1), device=cuda_device)
    th = torch.tensor([[float("nan"), 0, 0, 0, 1, 0], [1, 0, 0, 0, float("inf"), 0]], device=cuda_device)
    out = M.transformer(U, th, (5, 5))
    torch.cuda.synchronize()
    assert torch.isnan(out[0]).all()
    c = M.stn_corners(th, (9, 9), (5, 5))
    assert int(c.min()) >= 0 and int(c.max()) <= 8


def test_full_size_properties(cuda_device):
    """BASELINE config-5 size (B = 16384) through size-independent properties: linearity in U and in
    gout, zero gradient for out-of-range glimpses, determinism of the forward."""
    B = 16384
    g = torch.Generator(device=cuda_device).manual_seed(10)
    U = torch.rand((B, 50, 50, 1), device=cuda_device, generator=g)
    s, x, y = synth.sxy_prior_like(B, seed=1)
    th = torch.tensor(synth.theta_read(s, x, y), device=cuda_device)
    out1 = M.transformer(U, th, (28, 28))
    out2 = M.transformer(U, th, (28, 28))
    assert torch.equal(out1, out2)
    # exact linearity under power-of-two scaling (every product/sum scales exactly)
    assert torch.equal(M.transformer(U * 4.0, th, (28, 28)), out1 * 4.0)
    # checksum of checksums against the C oracle on a strided sample of the batch
    idx = torch.arange(0, B, 257, device=cuda_device)
    ref = RC.forward(U[idx].cpu().numpy(), th[idx].cpu().numpy(), (28, 28))
    assert H.same_bits_or_nan(out1[idx].cpu().numpy(), ref)
    # gradients: linear in gout
    Ug = U.clone().requires_grad_(True)
    tg = th.clone().requires_grad_(True)
    go = torch.randn((B, 28, 28, 1), device=cuda_device, generator=g)
    o = M.transformer(Ug, tg, (28, 28))
    dU1, dt1 = torch.autograd.grad(o, (Ug, tg), go, retain_graph=True)
    dU2, dt2 = torch.autograd.grad(o, (Ug, tg), go * 2.0)
    # (summation order may differ between launches: compare relative to the gradient scale)
    assert float((dU2 - dU1 * 2.0).abs().max()) <= 1e-4 * float(dU1.abs().max())
    assert float((dt2 - dt1 * 2.0).abs().max()) <= 1e-4 * float(dt1.abs().max())
    # sum(dU) == sum over in-range pixels of g (bilinear weights sum to 1): compare on the sample
    dUs, dts = R.transformer_backward(U[idx].cpu().numpy(), th[idx].cpu().numpy(), (28, 28), go[idx].cpu().numpy())
    aU, ath = R.backward_term_magnitudes(U[idx].cpu().numpy(), th[idx].cpu().numpy(), (28, 28), go[idx].cpu().numpy())
    assert H.grad_excess(dU1[idx].cpu().numpy(), dUs, aU) <= 1.0
    assert H.grad_excess(dt1[idx].cpu().numpy().reshape(-1, 2, 3), dts, ath) <= 1.0


def test_composite_golden(cuda_device):
    d = H.load("composite_28_50")
    dev = cuda_device
    canvas = torch.tensor(d["canvas"], device=dev, requires_grad=True)
    U = torch.tensor(d["U"], device=dev, requires_grad=True)
    th = torch.tensor(d["theta"], device=dev, requires_grad=True)
    z = torch.tensor(d["z"], device=dev, requires_grad=True)
    stop = torch.tensor(d["stop_sum"], device=dev)
    out = M.write_composite(canvas, U, th, z, stop, float(d["threshold"]))
    assert H.same_bits_or_nan(out.detach().cpu().numpy(), d["out"])
    out.backward(torch.tensor(d["gcanvas"], device=dev))
    assert np.array_equal(canvas.grad.cpu().numpy(), d["gcanvas"])
    mask = d["stop_sum"] < d["threshold"]
    gwin = (mask * d["z"])[:, None, None, None] * d["gcanvas"][..., None]
    aU, ath = R.backward_term_magnitudes(d["U"][..., None], d["theta"], (50, 50), gwin)
    assert H.grad_excess(U.grad.cpu().numpy()[..., None], d["dU"][..., None], aU) <= 1.0
    assert H.grad_excess(th.grad.cpu().numpy().reshape(-1, 2, 3), d["dtheta"], ath) <= 1.0
    win = R.transformer(d["U"][..., None], d["theta"], (50, 50))[..., 0]
    az = (np.abs(d["gcanvas"]) * np.abs(win)).sum((1, 2))
    assert H.grad_excess(z.grad.cpu().numpy(), d["dz"], az + 1e-3) <= 1.0
    # in-place form gives the same canvas and leaves inactive images untouched
    c2 = torch.tensor(d["canvas"], device=dev)
    r = M.write_composite(c2, U.detach(), th.detach(), z.detach(), stop, float(d["threshold"]), inplace=True)
    assert r.data_ptr() == c2.data_ptr()
    assert H.same_bits_or_nan(c2.cpu().numpy(), d["out"])
    # flat [B, cs*cs] canvases and windows like the reference's running_recon / vae_recon
    r2 = M.write_composite(torch.tensor(d["canvas"], device=dev).reshape(8, -1), U.detach().reshape(8, -1),
                           th.detach(), z.detach(), stop, float(d["threshold"]))
    assert r2.shape == (8, 2500) and H.same_bits_or_nan(r2.cpu().numpy().reshape(8, 50, 50), d["out"])


def test_composite_equals_unfused_ops(cuda_device):
    """Fused kernel == transformer() followed by the reference's where/mul/add (air_number_bbox_location.py:722-727)."""
    dev = cuda_device
    B = 256
    gen = torch.Generator(device=dev).manual_seed(2)
    canvas = torch.rand((B, 64, 64), device=dev, generator=gen)
    U = torch.sigmoid(torch.randn((B, 28, 28), device=dev, generator=gen))
    s, x, y = synth.sxy_prior_like(B, seed=9)
    th = torch.tensor(synth.theta_write(s, x, y), device=dev)
    z = torch.rand(B, device=dev, generator=gen)
    stop = torch.rand(B, device=dev, generator=gen) * 1.5
    fused = M.write_composite(canvas, U, th, z, stop, 0.9)
    win = M.transformer(U[..., None], th, (64, 64))[..., 0]
    unfused = canvas + torch.where((stop < 0.9)[:, None, None], z[:, None, None] * win, torch.zeros_like(win))
    assert torch.equal(fused, unfused)


@pytest.mark.parametrize("canvas,glimpse,direction", [(50, 28, "write"), (256, 64, "read"), (256, 64, "write")])
def test_full_size_properties_other_cells(cuda_device, canvas, glimpse, direction):
    """BASELINE config-5 batch (16384) at the headline cell and in the write direction, through size-independent
    properties: run-to-run determinism (forward and the gather-form backward), exact power-of-two linearity,
    parity with the C oracle on a strided sample of the batch (forward bit-exact, gradients within GRAD_RTOL)."""
    B = 16384
    gen = torch.Generator(device=cuda_device).manual_seed(canvas + glimpse)
    s, x, y = synth.sxy_prior_like(B, seed=3)
    if direction == "read":
        U = torch.rand((B, canvas, canvas, 1), device=cuda_device, generator=gen)
        th, out_size = torch.tensor(synth.theta_read(s, x, y), device=cuda_device), (glimpse, glimpse)
    else:
        U = torch.rand((B, glimpse, glimpse, 1), device=cuda_device, generator=gen)
        th, out_size = torch.tensor(synth.theta_write(s, x, y), device=cuda_device), (canvas, canvas)
    go = torch.randn((B, out_size[0], out_size[1], 1), device=cuda_device, generator=gen)
    Ug, tg = U.clone().requires_grad_(True), th.clone().requires_grad_(True)
    out = M.transformer(Ug, tg, out_size)
    dU1, dt1 = torch.autograd.grad(out, (Ug, tg), go, retain_graph=True)
    dU2, dt2 = torch.autograd.grad(out, (Ug, tg), go)
    assert torch.equal(dU1, dU2) and torch.equal(dt1, dt2), "separable thetas: the backward is atomic-free and deterministic"
    assert torch.equal(M.transformer(U * 0.5, th, out_size), out.detach() * 0.5)
    idx = torch.arange(0, B, 1021, device=cuda_device)
    Us, ts, gs_ = U[idx].cpu().numpy(), th[idx].cpu().numpy(), go[idx].cpu().numpy()
    assert H.same_bits_or_nan(out.detach()[idx].cpu().numpy(), RC.forward(Us, ts, out_size))
    dUs, dts = R.transformer_backward(Us, ts, out_size, gs_)
    aU, ath = R.backward_term_magnitudes(Us, ts, out_size, gs_)
    assert H.grad_excess(dU1[idx].cpu().numpy(), dUs, aU) <= 1.0
    assert H.grad_excess(dt1[idx].cpu().numpy().reshape(-1, 2, 3), dts, ath) <= 1.0


def test_host_buffer_entry_point_matches_device_path(cuda_device):
    """mog_stn_fwd_bwd_host (the end-to-end leg of bench.py): pinned host arrays in/out, chunked over streams --
    same bits as the device-resident calls, including a ragged last chunk and the dtheta-only form."""
    from mog_asr_b200.host_api import HostSampler
    rng = np.random.default_rng(77)
    B = 1000                                    # chunk 256 -> three full chunks and a ragged one
    U = torch.from_numpy(rng.random((B, 50, 50, 1), dtype=np.float32)).pin_memory()
    s, x, y = synth.sxy_prior_like(B, seed=8)
    th = torch.from_numpy(synth.theta_read(s, x, y)).pin_memory()
    g = torch.from_numpy(rng.standard_normal((B, 28, 28, 1), dtype=np.float32)).pin_memory()
    hs = HostSampler(cuda_device, (50, 50), (28, 28), 1, chunk=256, nstreams=3)
    out, dU, dth = hs.fwd_bwd(U, th, g)
    Ud, td = U.to(cuda_device).requires_grad_(True), th.to(cuda_device).requires_grad_(True)
    o = M.transformer(Ud, td, (28, 28))
    o.backward(g.to(cuda_device))
    assert torch.equal(out, o.detach().cpu()) and torch.equal(dU, Ud.grad.cpu()) and torch.equal(dth, td.grad.cpu())
    out2, dU2, dth2 = hs.fwd_bwd(U, th, g, need_dU=False)
    assert dU2 is None and torch.equal(out2, out) and torch.equal(dth2, dth)


@pytest.mark.gpu
def test_batch_host_entry_point_matches_batch_transformer(cuda_device):
    """mog_stn_batch_fwd_bwd_host: the batch_transformer form on host buffers (every source image uploaded once for its T
    transforms, dU summed over them) -- same bits as batch_transformer + autograd on the device, ragged last chunk, and the
    dtheta-only form of the AIR read site."""
    from mog_asr_b200.host_api import HostSampler
    rng = np.random.default_rng(78)
    B, T = 150, 4                                # chunk 64 -> two full chunks and a ragged one
    U = torch.from_numpy(rng.random((B, 50, 50, 1), dtype=np.float32)).pin_memory()
    s, x, y = synth.sxy_prior_like(B * T, seed=9)
    th = torch.from_numpy(synth.theta_read(s, x, y).reshape(B, T, 6)).pin_memory()
    g = torch.from_numpy(rng.standard_normal((B, T, 28, 28, 1), dtype=np.float32)).pin_memory()
    hs = HostSampler(cuda_device, (50, 50), (28, 28), 1, chunk=64, nstreams=3, transforms=T)
    out, dU, dth = hs.batch_fwd_bwd(U, th, g)
    Ud, td = U.to(cuda_device).requires_grad_(True), th.to(cuda_device).requires_grad_(True)
    o = M.batch_transformer(Ud, td, (28, 28))
    o.backward(g.reshape(B * T, 28, 28, 1).to(cuda_device))
    assert torch.equal(out, o.detach().cpu()) and torch.equal(dU, Ud.grad.cpu()) and torch.equal(dth, td.grad.cpu())
    out2, dU2, dth2 = hs.batch_fwd_bwd(U, th, g, need_dU=False)
    assert dU2 is None and torch.equal(out2, out) and torch.equal(dth2, dth)
    out3, dU3, dth3 = hs.batch_fwd_bwd(U, th)    # forward only
    assert dU3 is None and dth3 is None and torch.equal(out3, out)


@pytest.mark.gpu
@pytest.mark.parametrize("ws,cs,B,T,chunk", [(28, 50, 150, 3, 64), (64, 256, 70, 4, 32)])
def test_write_composite_host_entry_point_matches_the_device_loop(cuda_device, ws, cs, B, T, chunk):
    """mog_stn_write_composite_host: T windows per image composited onto one canvas per image from step-major host arrays,
    canvas gradient differentiated back to every step -- same bits as T device calls of write_composite + autograd
    (reference loop :592-600, :718-727), ragged last chunk, forward-only and partial-gradient forms; and the first step
    against the numpy oracle."""
    from mog_asr_b200.host_api import HostCompositeWriter
    rng = np.random.default_rng(ws + cs)
    W = torch.from_numpy(rng.random((T, B, ws, ws), dtype=np.float32)).pin_memory()
    s, x, y = synth.sxy_prior_like(T * B, seed=12)
    th = torch.from_numpy(synth.theta_write(s, x, y).reshape(T, B, 6)).pin_memory()
    z = torch.from_numpy(rng.random((T, B), dtype=np.float32)).pin_memory()
    g = torch.from_numpy(rng.standard_normal((B, cs, cs), dtype=np.float32)).pin_memory()
    hw = HostCompositeWriter(cuda_device, (ws, ws), (cs, cs), steps=T, chunk=chunk, nstreams=3)
    canvas, dW, dth, dz = hw.fwd_bwd(W, th, z, g)
    Wd, td, zd = (t.to(cuda_device).requires_grad_(True) for t in (W, th, z))
    c = torch.zeros((B, cs, cs), device=cuda_device)
    for t in range(T):
        c = M.write_composite(c, Wd[t], td[t], zd[t])
    c.backward(g.to(cuda_device))
    assert torch.equal(canvas, c.detach().cpu())
    assert torch.equal(dW, Wd.grad.cpu()) and torch.equal(dth, td.grad.cpu()) and torch.equal(dz, zd.grad.cpu())
    c2, dW2, dth2, dz2 = hw.fwd_bwd(W, th, z)                      # forward only
    assert dW2 is None and dth2 is None and dz2 is None and torch.equal(c2, canvas)
    c3, dW3, dth3, dz3 = hw.fwd_bwd(W, th, z, g, need_dW=False)
    assert dW3 is None and torch.equal(dth3, dth) and torch.equal(dz3, dz)
    hw1 = HostCompositeWriter(cuda_device, (ws, ws), (cs, cs), steps=1, chunk=chunk, nstreams=2)
    c1 = hw1.fwd_bwd(W[:1].contiguous(), th[:1].contiguous(), z[:1].contiguous())[0].numpy()
    ref = R.transformer(W[0].numpy()[..., None], th[0].numpy(), (cs, cs))[..., 0] * z[0].numpy()[:, None, None]
    np.testing.assert_array_equal(c1, ref + np.float32(0.0))


@pytest.mark.gpu
@pytest.mark.parametrize("src,dst", [((131, 127), (33, 29)), ((33, 29), (131, 127)), ((256, 256), (64, 64)), ((64, 64), (256, 256)),
                                     ((90, 93), (90, 93))])
def test_large_images_every_element_written(cuda_device, src, dst):
    """Large outputs / source gradients are mostly zeros written by the bulk-copy engine (rows outside the footprint)
    and by ordinary stores (the footprint band): poison the allocator's blocks first so that an element nobody wrote
    shows up as NaN; odd widths put every image at a different 16-byte misalignment."""
    B = 9
    rng = np.random.default_rng(src[0] * 7 + dst[1])
    s, x, y = synth.sxy_prior_like(B, seed=5)
    s[0], x[0], y[0] = 0.05, 0.97, -0.97          # footprint hanging over a corner
    s[1], x[1], y[1] = 1.7, 0.0, 0.0              # covers everything
    th = synth.theta_read(s, x, y) if src[0] >= dst[0] else synth.theta_write(s, x, y)
    th[2] = [0.5, 0, 5.0, 0, 0.5, 5.0]            # entirely out of range: no footprint at all
    U = rng.random((B, src[0], src[1], 1), dtype=np.float32)
    g = rng.normal(size=(B, dst[0], dst[1], 1)).astype(np.float32)
    for n in (B * src[0] * src[1], B * dst[0] * dst[1]):
        poison = torch.full((n,), float("nan"), device=cuda_device)
        del poison
    out, dU, dth = run_fwd_bwd(cuda_device, U, th, dst, g)
    ref_out = RC.forward(U, th, dst)
    assert H.same_bits_or_nan(out, ref_out)
    dU64, dth64 = R.transformer_backward(U, th, dst, g, dtype=np.float64)
    aU, ath = R.backward_term_magnitudes(U, th, dst, g)
    assert np.isfinite(dU).all()
    assert H.grad_excess(dU, dU64, aU) <= 1.0
    assert H.grad_excess(dth, dth64, ath) <= 1.0


def test_attention_boxes_match_oracle(cuda_device):
    """Visualisation consumer (air_number_bbox_location.py:243-288): frame template written through the backward ST
    matrices at 2x canvas resolution, clipped and thresholded; one shared template vs the oracle's physical copies."""
    n, steps, T, cs, ws, zoom = 5, 2, 3, 50, 28, 2
    s, x, y = synth.sxy_prior_like(n * steps, seed=8)
    th = synth.theta_write(s, x, y).reshape(n, steps, 6)
    got = M.attention_boxes(torch.tensor(th, device=cuda_device), cs, zoom=zoom, windows_size=ws, max_steps=T).cpu().numpy()
    tmpl = np.zeros((ws, ws, 1), np.float32)
    tmpl[0], tmpl[-1], tmpl[:, 0], tmpl[:, -1] = 1, 1, 1, 1
    thp = np.concatenate([th, np.zeros((n, T - steps, 6), np.float32)], 1).reshape(n * T, 6)
    ref = RC.forward(np.repeat(tmpl[None], n * T, 0), thp, (zoom * cs, zoom * cs))
    ref = (np.clip(ref, 0, 1) > 0.01).astype(np.float32).reshape(n, T, zoom * cs, zoom * cs)
    assert got.shape == ref.shape and np.array_equal(got, ref)
    assert 0 < got[:, :steps].mean() < 0.5          # frames, not filled boxes
    assert np.all(got[:, steps:] == 0.0)            # zero matrices sample the template's centre (= 0) everywhere


@pytest.mark.parametrize("name", ["read_50_28", "write_28_50", "adversarial_17x23x3_9x31", "adversarial_50_28", "adversarial_28_50",
                                  "out_1x1", "out_1x7", "fullcover_64_28"])
def test_forward_equals_the_reference_source_run_on_the_tf_shim(cuda_device, name):
    """CUDA forward against ``tests/golden/graph_*.npz``: the outputs of the reference's own ``air/transformer.py``
    executed on the numpy TF shim (see tests/test_oracle.py) -- bit for bit."""
    import os
    here = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    z, g = np.load(os.path.join(here, name + ".npz")), np.load(os.path.join(here, "graph_" + name + ".npz"))
    rows = g["rows"]
    out = M.transformer(torch.tensor(z["U"][rows], device=cuda_device), torch.tensor(z["theta"][rows], device=cuda_device),
                        tuple(int(v) for v in z["out_size"])).cpu().numpy()
    assert np.array_equal(out.view(np.uint32), g["out"].view(np.uint32))


def test_batch_transformer_equals_the_reference_source_run_on_the_tf_shim(cuda_device):
    import os
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "graph_batch_transformer.npz"))
    out = M.batch_transformer(torch.tensor(g["U"], device=cuda_device), torch.tensor(g["thetas"], device=cuda_device),
                              tuple(g["out"].shape[1:3])).cpu().numpy()
    assert np.array_equal(out.view(np.uint32), g["out"].view(np.uint32))


@pytest.mark.parametrize("name", ["read_50_28", "write_28_50", "adversarial_17x23x3_9x31", "fullcover_64_28", "out_1x7"])
def test_backward_matches_autodiff_of_the_reference_source(cuda_device, name):
    """CUDA gradients against ``tests/golden/graph_grad_*.npz`` (autograd of the reference's own graph on the torch TF shim,
    float32): both are fp32 evaluations in different summation orders, so each gets half of the tolerance budget around
    the fp64 closed form -- asserted directly against each other with 2 x GRAD_RTOL."""
    import os
    here = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    z, g = np.load(os.path.join(here, name + ".npz")), np.load(os.path.join(here, "graph_grad_" + name + ".npz"))
    rows = g["rows"]
    _, dU, dth = run_fwd_bwd(cuda_device, z["U"][rows], z["theta"][rows], z["out_size"], z["gout"][rows])
    assert H.grad_excess(dU, g["dU"], z["absdU"][rows], rtol=2 * H.GRAD_RTOL) <= 1.0
    assert H.grad_excess(dth, g["dtheta"], z["absdtheta"][rows], rtol=2 * H.GRAD_RTOL) <= 1.0


@pytest.mark.gpu
@pytest.mark.parametrize("Hs,Ws,Ho,Wo,B,full", [
    (28, 28, 50, 50, 33, False), (64, 64, 256, 256, 9, True), (64, 64, 256, 256, 9, False), (50, 50, 28, 28, 33, False),
    (64, 64, 128, 128, 17, True), (256, 256, 64, 64, 13, False), (256, 256, 64, 64, 13, True),
    (32, 32, 20, 20, 33, False),     # read with Ws <= 32: one source-column chunk per streaming pass
    (96, 96, 128, 128, 9, False),    # write with Ws > 64: streaming, dU outside the footprint zeroed by the bulk-copy engine
    (64, 64, 48, 256, 9, False)])    # wide output shorter than the source: streaming
def test_separable_backward_meets_the_gradient_contract(cuda_device, Hs, Ws, Ho, Wo, B, full):
    """The separable backward through the theta-taking entry point, dU and dtheta pre-filled with NaN: the source-column kernel
    (output at least as large as the source) and the streaming kernel (everything else), at every source-width class that
    selects a different instantiation, meet the fp64-oracle tolerance in both directions."""
    L = _lib.load()
    rng = np.random.default_rng(Hs + Ho)
    U = rng.random((B, Hs, Ws, 1), dtype=np.float32)
    s, x, y = synth.sxy_full_cover(B, seed=3) if full else synth.sxy_prior_like(B, seed=3)
    th = synth.theta_read(s, x, y) if Ws > Wo else synth.theta_write(s, x, y)
    g = rng.normal(size=(B, Ho, Wo, 1)).astype(np.float32)
    dU = torch.full((B, Hs, Ws, 1), float("nan"), device=cuda_device)
    dth = torch.full((B, 6), float("nan"), device=cuda_device)
    Ud, thd, gd = (torch.tensor(a, device=cuda_device) for a in (U, th, g))
    rc = L.mog_stn_backward(Ud.data_ptr(), thd.data_ptr(), gd.data_ptr(), dU.data_ptr(), dth.data_ptr(), B, Hs, Ws, 1, Ho, Wo, 1, None)
    torch.cuda.synchronize()
    assert rc == 0, _lib.last_error()
    rU, rth = R.transformer_backward(U, th, (Ho, Wo), g)
    aU, ath = R.backward_term_magnitudes(U, th, (Ho, Wo), g)
    assert H.grad_excess(dU.cpu().numpy(), rU, aU) <= 1.0
    assert H.grad_excess(dth.cpu().numpy().reshape(-1, 2, 3), rth, ath) <= 1.0


@pytest.mark.gpu
@pytest.mark.parametrize("cs,ws,B", [(50, 28, 300), (256, 64, 24),
                                     # glimpse larger than the canvas, canvas <= 32 or window > 64: together with the two cells
                                     # above, every source-width class of both backward kernels in both directions
                                     (20, 28, 64), (50, 64, 32), (32, 20, 64), (128, 96, 16)])
def test_sxy_entry_points_equal_the_theta_path(cuda_device, cs, ws, B):
    """Theta built inside the sampler kernels from the model's (s, x, y) (SURVEY 8(f)2; reference :511-531, :563-584): the read
    and the write + composite give the same bits as the theta-taking entry points fed by the theta kernel, and d_shift /
    d_scale -- the write call's share added inside the read call's backward kernel -- equal autograd through the theta
    kernel within the gradient tolerance."""
    from mog_asr_b200.air.fused import thetas
    from mog_asr_b200.sxy import read_glimpse_sxy, write_composite_sxy
    rng = np.random.default_rng(cs + ws)
    s, x, y = synth.sxy_prior_like(B, seed=21)
    img = torch.tensor(rng.random((B, cs, cs, 1), dtype=np.float32), device=cuda_device)
    win = torch.tensor(rng.random((B, ws, ws), dtype=np.float32), device=cuda_device)
    z = torch.tensor(rng.random(B, dtype=np.float32), device=cuda_device)
    stop = torch.tensor(rng.random(B, dtype=np.float32) * 1.2, device=cuda_device)       # some images inactive (>= 0.9)
    canvas0 = torch.tensor(rng.random((B, cs, cs), dtype=np.float32), device=cuda_device)
    g_win = torch.tensor(rng.standard_normal((B, ws, ws, 1), dtype=np.float32), device=cuda_device)
    g_can = torch.tensor(rng.standard_normal((B, cs, cs), dtype=np.float32), device=cuda_device)

    def leaves():
        sh = torch.tensor(np.stack([x, y], 1).astype(np.float32), device=cuda_device, requires_grad=True)
        sc = torch.tensor(s.astype(np.float32)[:, None], device=cuda_device, requires_grad=True)
        return sh, sc, win.clone().requires_grad_(True), z.clone().requires_grad_(True)

    sh1, sc1, w1, z1 = leaves()                                  # theta path
    th_r, th_w = thetas(sh1, sc1)
    out1 = M.transformer(img, th_r, (ws, ws))
    can1 = M.write_composite(canvas0, w1, th_w, z1, stop, 0.9)
    ((out1 * g_win).sum() + (can1 * g_can).sum()).backward()
    sh2, sc2, w2, z2 = leaves()                                  # theta in the kernels
    out2, shp, scp = read_glimpse_sxy(img, sh2, sc2, (ws, ws))
    can2 = write_composite_sxy(canvas0, w2, shp, scp, z2, stop, 0.9)
    ((out2 * g_win).sum() + (can2 * g_can).sum()).backward()
    assert torch.equal(out1, out2) and torch.equal(can1, can2)
    assert torch.equal(w1.grad, w2.grad) and torch.equal(z1.grad, z2.grad)
    for a, b in ((sh1.grad, sh2.grad), (sc1.grad, sc2.grad)):
        scale = float(a.abs().max())
        assert float((a - b).abs().max()) <= 2e-5 * scale, (float((a - b).abs().max()), scale)
    # the write call alone (nothing added in) and the read call alone
    sh3, sc3, w3, z3 = leaves()
    write_composite_sxy(canvas0, w3, sh3, sc3, z3, stop, 0.9).backward(g_can)
    sh4, sc4, w4, z4 = leaves()
    _, th_w4 = thetas(sh4, sc4)
    M.write_composite(canvas0, w4, th_w4, z4, stop, 0.9).backward(g_can)
    assert float((sh3.grad - sh4.grad).abs().max()) <= 2e-5 * float(sh4.grad.abs().max())
    assert float((sc3.grad - sc4.grad).abs().max()) <= 2e-5 * float(sc4.grad.abs().max())
