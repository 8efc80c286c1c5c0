"""The reference's trip count in the fixed-trip-count step, on the GPU: the ``mog_asr_reg_*_steps`` kernels against the plain ASR
kernels on the executed columns (bit for bit), the training step with the product operators against the reference loop
(``while any(stop_sum < thr)``, air_number_bbox_location.py:386-390) at planted trip counts, the captured step following the
trip count from replay to replay, and the two-GPU data-parallel form."""
import ctypes
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from mog_asr_b200 import _lib
from mog_asr_b200.air import AIRModel, Trainer, config_from_flags
from oracle.air_ops import SeededNoise
from tests.test_asr_kernels_gpu import ALL_ON, GATES, c_config, colsum_pass, excess, sigmoid64
from tests.test_reference_trip_count import C2, C3, DP_B, DP_TRIPS, PlantedTrips, make_images, planted

pytestmark = pytest.mark.gpu

GAMMA_SETS = {"all_on": ALL_ON, **GATES}
NCOMP = _lib.MOG_ASR_NUM_COMPONENTS


def mse(x, r):
    return ((x - r) ** 2).sum(1) * 50.0


def launch(fn, *args):
    rc = fn(*args, torch.cuda.current_stream().cuda_stream)
    assert rc == 0, _lib.last_error()


def nan(*shape, dev):
    return torch.full(shape, float("nan"), device=dev)


def forward(L, steps, lo, sh, sc, psum, inv_B, cfg, dev):
    """NaN-filled outputs; the *_steps form also returns its steps_out (NaN bits, -1, before the call)"""
    B, T = lo.shape
    per_image, comps, margin = nan(B, dev=dev), nan(B, NCOMP, dev=dev), nan(1, dev=dev)
    if not steps:
        launch(L.mog_asr_reg_forward, lo.data_ptr(), sh.data_ptr(), sc.data_ptr(), psum.data_ptr(), inv_B, B, T, ctypes.byref(cfg),
               per_image.data_ptr(), comps.data_ptr(), margin.data_ptr())
        return per_image, comps, margin
    n = torch.full((1,), -1, dtype=torch.int32, device=dev)
    launch(L.mog_asr_reg_forward_steps, lo.data_ptr(), sh.data_ptr(), sc.data_ptr(), psum.data_ptr(), inv_B, B, T,
           ctypes.byref(cfg), per_image.data_ptr(), comps.data_ptr(), margin.data_ptr(), n.data_ptr())
    return per_image, comps, margin, n


def backward(L, steps, lo, sh, sc, psum, inv_B, gp, gm, cfg, dev):
    B, T = lo.shape
    d_lo, d_sh, d_sc = nan(B, T, dev=dev), nan(B, T, 2, dev=dev), nan(B, T, dev=dev)
    fn = L.mog_asr_reg_backward_steps if steps else L.mog_asr_reg_backward
    launch(fn, lo.data_ptr(), sh.data_ptr(), sc.data_ptr(), psum.data_ptr(), inv_B, gp.data_ptr(), gm.data_ptr(), B, T,
           ctypes.byref(cfg), d_lo.data_ptr(), d_sh.data_ptr(), d_sc.data_ptr())
    return d_lo, d_sh, d_sc


def colsum_steps(L, lo, active, psum):
    B, T = lo.shape
    launch(L.mog_asr_reg_colsum_steps, lo.data_ptr(), active.data_ptr(), psum.data_ptr(), B, T)


def random_inputs(B, T, g, dev):
    lo = (torch.randn(B, T, generator=g, device=dev) * 2.0).clamp(-7.0, 7.0)
    sh = torch.tanh(torch.randn(B, T, 2, generator=g, device=dev) * 0.8)
    sc = torch.sigmoid(torch.randn(B, T, generator=g, device=dev) * 0.6 - 1.0)
    gp = torch.randn(B, generator=g, device=dev)
    return lo, sh, sc, gp


def planted_active(B, T, k, g, dev):
    """[T][B] bytes: image b is active after steps t < trips[b] - 1, trips in [1, k], one image at exactly k"""
    trips = torch.randint(1, k + 1, (B,), generator=g, device=dev)
    trips[int(torch.randint(0, B, (1,), generator=g, device=dev))] = k
    return (torch.arange(T, device=dev)[:, None] < trips[None, :] - 1).to(torch.uint8).contiguous()


def check_against_plain(L, dev, lo, sh, sc, gp, gm, psum, inv_B, cfg, k):
    """the *_steps forward / backward over T columns with psum [2T] against the plain kernels on contiguous copies of the
    first k columns with psum[0:k): the same bits; gradient columns >= k exactly 0; steps_out == k"""
    T = lo.shape[1]
    cut = [x[:, :k].contiguous() for x in (lo, sh, sc)]
    got = forward(L, True, lo, sh, sc, psum, inv_B, cfg, dev)
    ref = forward(L, False, *cut, psum[:k], inv_B, cfg, dev)
    for a, b in zip(got[:3], ref):
        assert torch.equal(a, b)
    assert int(got[3]) == k
    gd = backward(L, True, lo, sh, sc, psum, inv_B, gp, gm, cfg, dev)
    rd = backward(L, False, *cut, psum[:k], inv_B, gp, gm, cfg, dev)
    for a, b in zip(gd, rd):
        assert torch.equal(a[:, :k], b)
        assert torch.equal(a[:, k:], torch.zeros_like(a[:, k:])), "columns past the trip count"
    assert T >= k
    return got, gd


@pytest.mark.parametrize("B", [1, 127, 128, 129, 4097])
def test_steps_kernels_equal_the_plain_kernels_on_the_executed_columns(cuda_device, B):
    """Every T from 1 to 16 and every planted trip count k <= T through the active stack, under every gamma combination of the
    gate tests: the column sum counts exactly and keeps the plain column sum's P bound; forward (per_image, components, margin)
    and backward equal the plain kernels' bits on the first k columns, later gradient columns are exactly 0, steps_out == k."""
    L, dev = _lib.load(), cuda_device
    g = torch.Generator(device=dev).manual_seed(B)
    gm = torch.tensor([0.7], device=dev)
    per_pass = colsum_pass(dev)
    depth = 3 + -(-B // per_pass) + 5 + per_pass // 32
    for T in range(1, _lib.MOG_ASR_MAX_STEPS + 1):
        lo, sh, sc, gp = random_inputs(B, T, g, dev)
        P64 = sigmoid64(lo.cpu().numpy().astype(np.float64)).sum(0)
        for k in range(1, T + 1):
            active = planted_active(B, T, k, g, dev)
            psum = torch.zeros(2 * T, device=dev)
            colsum_steps(L, lo, active, psum)
            assert torch.equal(psum[T:], active.sum(1).to(torch.float32))
            assert excess(psum[:T].cpu().numpy(), P64, depth * P64, ulps=2) <= 1.0
            for name, gam in GAMMA_SETS.items():
                cfg = c_config(dict(canvas_size=50.0, counts=[1, 2, 4], max_steps=T, area_minmax=(11.0, 15.0), **gam))
                check_against_plain(L, dev, lo, sh, sc, gp, gm, psum, np.float32(1.0 / B).item(), cfg, k)


def test_steps_kernels_on_shards(cuda_device):
    """Shards of 100 and 157 images whose local batches would stop after step 1 and after step 3: their [2T] psums summed (as
    the all-reduce does) give both shards 4 steps and, concatenated, the bits of the whole-batch call with that psum."""
    L, dev = _lib.load(), cuda_device
    T, B = 6, 257
    g = torch.Generator(device=dev).manual_seed(257)
    lo, sh, sc, gp = random_inputs(B, T, g, dev)
    gm = torch.tensor([0.7], device=dev)
    parts = [slice(0, 100), slice(100, 257)]
    active = torch.cat([planted_active(100, T, 2, g, dev), planted_active(157, T, 4, g, dev)], 1).contiguous()
    psum = torch.zeros(2 * T, device=dev)
    for s in parts:
        p = torch.zeros(2 * T, device=dev)
        colsum_steps(L, lo[s].contiguous(), active[:, s].contiguous(), p)
        assert float(p[T + (1 if s.start == 0 else 3)]) == 0.0
        psum += p
    assert torch.equal(psum[T:], active.sum(1).to(torch.float32))
    cfg = c_config(dict(canvas_size=50.0, counts=[1, 2, 4], max_steps=T, area_minmax=(11.0, 15.0), **ALL_ON))
    inv_B = np.float32(1.0 / B).item()
    whole_f, whole_b = check_against_plain(L, dev, lo, sh, sc, gp, gm, psum, inv_B, cfg, 4)
    for s in parts:
        x = [t[s].contiguous() for t in (lo, sh, sc, gp)]
        f, b = check_against_plain(L, dev, *x[:3], x[3], gm, psum, inv_B, cfg, 4)
        assert torch.equal(f[2], whole_f[2]) and int(f[3]) == 4
        for a, w in zip((f[0], f[1]) + b, (whole_f[0], whole_f[1]) + whole_b):
            assert torch.equal(a, w[s])


def test_zero_batch_forward_writes_margin_and_steps(cuda_device):
    """a rank without images still writes the margin (from the global psum) and the global trip count"""
    L, dev = _lib.load(), cuda_device
    T = 6
    psum = torch.tensor([40.0, 21.0, 9.0, 3.0, 1.0, 0.5] + [17.0, 5.0, 0.0, 2.0, 0.0, 0.0], device=dev)
    cfg = c_config(dict(canvas_size=50.0, counts=[1, 3], max_steps=T, area_minmax=(11.0, 15.0), **ALL_ON))
    empty = torch.empty(0, T, device=dev)
    got = forward(L, True, empty, torch.empty(0, T, 2, device=dev), empty, psum, 1.0 / 64, cfg, dev)
    ref = forward(L, False, torch.empty(0, 3, device=dev), torch.empty(0, 3, 2, device=dev), torch.empty(0, 3, device=dev),
                  psum[:3], 1.0 / 64, cfg, dev)
    assert int(got[3]) == 3 and torch.isfinite(got[2]).all() and float(got[2]) > 0
    assert torch.equal(got[2], ref[2])


# ---- the training step with the product operators -------------------------------------------------------------------
def assert_params_close(model, g_ref, g_got, rel=2e-3):
    off = 0
    for name, p in model.named_parameters():
        n = p.numel()
        a, b = g_ref[off:off + n].double(), g_got[off:off + n].double()
        off += n
        assert torch.isfinite(b).all(), name
        assert float((a - b).abs().max()) <= rel * float(a.abs().max()) + 1e-12, name


@pytest.mark.parametrize("flags", [C2, C3], ids=["C2", "C3"])
@pytest.mark.parametrize("k", [1, 2, 4, 6])
def test_product_step_equals_the_reference_loop(cuda_device, flags, k):
    """fp32, product operators on both sides, squared-error reconstruction, planted trip count k: the fixed-trip-count step with
    ``reference_trip_count`` (batched tail, fused kernels) against the reference loop with the same weights and noise."""
    dev = cuda_device
    B = 12
    ref = Trainer(config_from_flags(always_max_steps=False, **flags), dev, seed=5)
    got = Trainer(config_from_flags(always_max_steps=True, reference_trip_count=True, **flags), dev, seed=5)
    got.model.load_state_dict(ref.model.state_dict())
    images = make_images(B, ref.cfg.canvas_size, seed=8).to(dev)
    noise = lambda: PlantedTrips(SeededNoise(3, B, device=dev), planted(k, B))
    o_ref = ref.forward_backward(images, noise=noise(), recon_loss_fn=mse)
    o_got = got.forward_backward(images, noise=noise(), recon_loss_fn=mse)
    assert o_ref["steps"] == k and int(o_got["steps"]) == k
    assert torch.equal(o_got["rec_num_digits"], o_ref["rec_num_digits"])
    np.testing.assert_allclose(float(o_got["loss"].detach()), float(o_ref["loss"].detach()), rtol=2e-5)
    assert_params_close(got.model, ref.flat_grad, got.flat_grad)


class _MseTrainer(Trainer):
    """the training step with the well-conditioned squared-error reconstruction (captured as well)"""

    def forward_backward(self, images, noise=None, recon_loss_fn=None):
        return super().forward_backward(images, noise, recon_loss_fn=mse)


def test_captured_step_follows_the_trip_count(cuda_device):
    """One capture (C2 flags, B = 32); between replays the z_pres posterior's output bias is set in place so that the loop stops
    after step 0, never, and after a middle step: ``steps`` follows without a recapture.  The middle replay's draws, read from
    the trainer's noise bank (static graph memory), drive an eager reference-loop step from the same pre-replay parameters:
    the same trip count, loss and (cleaned, clipped) gradients within the bounds of the product-step test."""
    dev = cuda_device
    B = 32
    cfg = config_from_flags(always_max_steps=True, reference_trip_count=True, **C2)
    images = make_images(B, 50, seed=12).to(dev)
    tr = _MseTrainer(cfg, dev, seed=21).capture(B)
    bias = tr.model.z_post.bias
    torch.cuda.manual_seed(777)
    for b, expect in ((-100.0, 1), (100.0, 6), (-100.0, 1)):
        with torch.no_grad():
            bias.fill_(b)
        out = tr.step_graph(images)
        torch.cuda.synchronize()
        assert int(out["steps"]) == expect, b
    with torch.no_grad():
        bias.fill_(-1.5)
    pre = {n: t.detach().clone() for n, t in tr.model.state_dict().items()}
    out = tr.step_graph(images)
    torch.cuda.synchronize()
    steps = int(out["steps"])
    assert 1 < steps < 6
    bank = {kind: t.clone() for kind, t in tr._noise_bank.items()}
    ref = _MseTrainer(config_from_flags(always_max_steps=False, **C2), dev, seed=21)
    ref.model.load_state_dict(pre)
    o_ref = ref.forward_backward(images, noise=lambda kind, step, shape: bank[kind][step])
    ref.clean_and_clip()
    assert o_ref["steps"] == steps
    assert torch.equal(out["rec_num_digits"], o_ref["rec_num_digits"])
    np.testing.assert_allclose(float(out["loss"].detach()), float(o_ref["loss"].detach()), rtol=2e-5)
    assert_params_close(ref.model, ref.flat_grad, tr.flat_grad)


# ---- two GPUs over NCCL ----------------------------------------------------------------------------------------------
def _nccl_worker(rank, world, port, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dev = torch.device("cuda", rank)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        lo, hi = rank * DP_B // world, (rank + 1) * DP_B // world
        images = make_images(DP_B, 50).to(dev)
        cfg = config_from_flags(always_max_steps=True, reference_trip_count=True, **C2)
        tr = Trainer(cfg, dev, process_group=dist.group.WORLD, global_batch=DP_B, seed=5)
        out = tr.forward_backward(images[lo:hi], noise=PlantedTrips(SeededNoise(7, DP_B, lo, hi, device=dev), DP_TRIPS),
                                  recon_loss_fn=mse)
        tr.reduce_gradients()
        ret[f"steps{rank}"] = int(out["steps"])
        if rank == 0:
            one = Trainer(config_from_flags(always_max_steps=False, **C2), dev, seed=5)
            o = one.forward_backward(images, noise=PlantedTrips(SeededNoise(7, DP_B, device=dev), DP_TRIPS), recon_loss_fn=mse)
            ret["steps_single"] = o["steps"]
            ret["flat_grad"], ret["flat_grad_single"] = tr.flat_grad.cpu(), one.flat_grad.cpu()
    finally:
        dist.destroy_process_group()


def test_data_parallel_ranks_stopping_at_different_steps_nccl(cuda_device):
    """The gloo test's form with the product operators on two GPUs: both ranks run the global batch's 4 steps, and the
    all-reduced gradient equals the single-process reference-loop gradient of the whole batch."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ret = mp.Manager().dict()
    mp.spawn(_nccl_worker, args=(2, port, ret), nprocs=2, join=True)
    assert ret["steps0"] == ret["steps1"] == ret["steps_single"] == 4
    assert_params_close(AIRModel(config_from_flags(**C2)), ret["flat_grad_single"], ret["flat_grad"])
