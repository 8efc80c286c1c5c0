"""The captured step with the reference's trip count (``AIRConfig.reference_trip_count``), on the CPU: the step that always
runs ``max_steps`` iterations but trains the reference loop's objective, with the oracle's operators in float64, against the
reference loop itself (``while any(stop_sum < thr)``, air_number_bbox_location.py:386-390) at planted trip counts; the
data-parallel form over gloo with ranks whose local batches stop at different steps; and the argument checks of the three
new entry points (``mog_asr_reg_*_steps``)."""
import ctypes
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from mog_asr_b200 import _lib, build, synth
from mog_asr_b200.air import Trainer, config_from_flags
from oracle.air_ops import OracleOps, SeededNoise

C2 = dict(data="mnist", dn="13", gm=100.0, gne=10.0)
C3 = dict(data="sprites", dn="3", ds="bbox20k", gb=1.0, gs=10.0, ga=20.0)


class ExecutedOracleOps(OracleOps):
    """The oracle's operators with the executed-steps form of the regularisers that ``AIRConfig.reference_trip_count`` asks
    of ``ops.asr``: with ``active [T, B]`` given, the trip count of the reference loop (``:386-390``) is taken as a host value
    from the active counts over the global batch (all-reduced under a process group), ``asr_terms`` sees only the first
    ``steps`` columns, so autograd gives the rest zero gradients, and ``steps`` (0-d int32) is returned as a 4th result."""

    def asr(self, cfg, log_odds, shifts, scales, active=None):
        if active is None:
            return super().asr(cfg, log_odds, shifts, scales)
        count = active.to(torch.float64).sum(1)                           # active images after each step
        if self.pg is not None:
            dist.all_reduce(count, group=self.pg)
        T = active.shape[0]
        Te = next((t + 1 for t in range(T - 1) if float(count[t]) == 0.0), T)
        per_image, margin, comps = super().asr(cfg, log_odds[:, :Te], shifts[:, :Te], scales[:, :Te])
        return per_image, margin, comps, torch.tensor(Te, dtype=torch.int32, device=log_odds.device)


def make_images(B, cs, seed=0):
    canv, _ = synth.multi_object_canvases(B, cs, 28, (1, 2, 3), seed=seed)
    return torch.tensor(np.clip(canv, 0, 1).reshape(B, cs * cs))


class PlantedTrips:
    """``SeededNoise`` whose Concrete draw is ``u = 1 - 1e-4`` before an image's planned last step and ``1e-4`` from it on.  At
    initialisation ``u = 1e-4`` gives z_pres ~ 0, so the stopping sum passes 0.9 and the image stops; image ``b`` is active
    for exactly ``trips[b]`` steps, and the reference loop runs ``max(trips)`` iterations."""

    def __init__(self, base, trips):
        self.base, self.trips = base, torch.as_tensor(trips)[base.lo:base.hi]

    def __call__(self, kind, step, shape):
        x = self.base(kind, step, shape)
        if kind != "concrete":
            return x
        keep = (step < self.trips - 1).to(x.device)
        return torch.where(keep, torch.full_like(x, 1 - 1e-4), torch.full_like(x, 1e-4))


def planted(k, B):
    """trip counts 1, 2, ..., k, 1, 2, ... over the batch: the batch runs k steps, its images stop at every step up to k"""
    return [1 + b % k for b in range(B)]


def run_step(flags, k, B=6, seed=5, **mode):
    cfg = config_from_flags(**mode, **flags)
    images = make_images(B, cfg.canvas_size, seed=2)
    tr = Trainer(cfg, "cpu", ops=ExecutedOracleOps(), seed=seed, dtype=torch.float64)
    out = tr.forward_backward(images.double(), noise=PlantedTrips(SeededNoise(4, B, dtype=torch.float64), planted(k, B)))
    return out, tr.flat_grad.clone()


def assert_grads_close(g0, g1, rel):
    fin = torch.isfinite(g0)
    assert torch.equal(torch.isfinite(g1), fin)
    assert float(g0[fin].abs().max()) > 0
    assert float((g1[fin] - g0[fin]).abs().max()) <= rel * float(g0[fin].abs().max())


def test_reference_trip_count_needs_always_max_steps():
    with pytest.raises(ValueError, match="always_max_steps"):
        config_from_flags(reference_trip_count=True, **C2)
    assert config_from_flags(always_max_steps=True, reference_trip_count=True, **C2).reference_trip_count


@pytest.mark.parametrize("flags", [C2, C3], ids=["C2", "C3"])
@pytest.mark.parametrize("k", [1, 2, 4, 6])
def test_executed_steps_equal_the_reference_loop(flags, k):
    """Float64 oracle operators, same weights and noise, planted trip count k: the fixed-trip-count step with
    ``reference_trip_count`` (batched tail) against the reference loop.  Same trip count, digit counts and canvas; loss, per-image
    ELBO and every finite gradient within the bounds of the batched-tail-vs-loop parity (GEMM row batching and the order of
    the sums over steps differ).  The extra iterations past k contribute exact zeros."""
    ref, g_ref = run_step(flags, k, always_max_steps=False)
    got, g_got = run_step(flags, k, always_max_steps=True, reference_trip_count=True)
    assert ref["steps"] == k
    assert got["steps"].dtype == torch.int32 and got["steps"].dim() == 0 and int(got["steps"]) == k
    assert torch.equal(got["rec_num_digits"], ref["rec_num_digits"])
    assert torch.allclose(got["reconstruction"], ref["reconstruction"], atol=1e-6)
    np.testing.assert_allclose(float(got["loss"].detach()), float(ref["loss"].detach()), rtol=1e-8)
    assert torch.allclose(got["elbo"], ref["elbo"], rtol=1e-8, atol=1e-4)
    np.testing.assert_allclose(got["per_image_reg"].numpy(), ref["per_image_reg"].numpy(), rtol=1e-8, atol=1e-10)
    np.testing.assert_allclose(float(got["margin"]), float(ref["margin"]), rtol=1e-8, atol=1e-12)
    # the logged per-step outputs keep max_steps columns; the first k are the reference loop's
    assert got["z_pres_probs"].shape[1] == 6 and ref["z_pres_probs"].shape[1] == k
    np.testing.assert_allclose(got["z_pres_probs"][:, :k].numpy(), ref["z_pres_probs"].numpy(), rtol=1e-8, atol=1e-12)
    assert_grads_close(g_ref, g_got, 1e-4)
    if k == 6:   # the reference loop runs all iterations: the mode computes exactly what the fixed mode does
        fixed, g_fixed = run_step(flags, k, always_max_steps=True)
        assert fixed["steps"] == 6
        assert torch.equal(got["loss"].detach(), fixed["loss"].detach())
        assert torch.equal(got["per_image_reg"], fixed["per_image_reg"]) and torch.equal(got["margin"], fixed["margin"])
        assert torch.equal(g_got, g_fixed)


# ---- data parallel over gloo ---------------------------------------------------------------------------------------
DP_B = 8
# rank 0 (images 0-3) stops after step 1, rank 1 (images 4-7) after step 3: the global batch runs 4 steps on both ranks
DP_TRIPS = [1, 2, 2, 1, 4, 3, 1, 4]


def _dp_worker(rank, world, port, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        cfg = config_from_flags(always_max_steps=True, reference_trip_count=True, **C2)
        images = make_images(DP_B, 50).double()
        lo, hi = rank * DP_B // world, (rank + 1) * DP_B // world
        tr = Trainer(cfg, "cpu", process_group=dist.group.WORLD, global_batch=DP_B, dtype=torch.float64,
                     ops=ExecutedOracleOps(process_group=dist.group.WORLD, global_batch=DP_B))
        out = tr.forward_backward(images[lo:hi], noise=PlantedTrips(SeededNoise(7, DP_B, lo, hi, dtype=torch.float64), DP_TRIPS))
        tr.reduce_gradients()
        ret[f"steps{rank}"] = int(out["steps"])
        ret[f"local_steps{rank}"] = max(DP_TRIPS[lo:hi])
        if rank == 0:
            ret["flat_grad"] = tr.flat_grad.clone()
    finally:
        dist.destroy_process_group()


def test_data_parallel_ranks_stopping_at_different_steps_gloo():
    """Two gloo ranks whose local batches would stop after step 1 and after step 3: the trip count is the global batch's
    (the active counts are all-reduced with the column sums), both ranks report 4 steps, and the all-reduced gradient equals
    the single-process reference-loop gradient of the whole batch."""
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ret = mp.Manager().dict()
    mp.spawn(_dp_worker, args=(2, port, ret), nprocs=2, join=True)
    assert (ret["local_steps0"], ret["local_steps1"]) == (2, 4)
    assert ret["steps0"] == ret["steps1"] == 4
    cfg = config_from_flags(always_max_steps=False, **C2)
    tr = Trainer(cfg, "cpu", ops=ExecutedOracleOps(), dtype=torch.float64)
    out = tr.forward_backward(make_images(DP_B, 50).double(), noise=PlantedTrips(SeededNoise(7, DP_B, dtype=torch.float64), DP_TRIPS))
    assert out["steps"] == 4
    assert_grads_close(tr.flat_grad, ret["flat_grad"], 1e-4)


# ---- argument checks of the C entry points (host only) ---------------------------------------------------------------
@pytest.fixture(scope="module")
def lib():
    build.build()
    return _lib.load()


def test_bad_arguments_of_the_steps_entry_points(lib):
    one = 0x1000   # never dereferenced: validation fails first
    cfg = _lib.AsrConfig()
    cfg.num_counts, cfg.counts[0], cfg.counts[1], cfg.gamma_margin = 2, 1, 3, 1.0
    c = ctypes.byref(cfg)

    def colsum(B=4, T=6, lo=one, act=one, psum=one):
        return lib.mog_asr_reg_colsum_steps(lo, act, psum, B, T, None)

    def forward(B=4, T=6, ins=(one,) * 4, outs=(one, None, one, None), cfg_=c):
        return lib.mog_asr_reg_forward_steps(*ins, 0.25, B, T, cfg_, *outs, None)

    def backward(B=4, T=6, ins=(one,) * 4, grads=(one, one), outs=(one,) * 3, cfg_=c):
        return lib.mog_asr_reg_backward_steps(*ins, 0.25, *grads, B, T, cfg_, *outs, None)

    for fn in (colsum, forward, backward):
        for T in (0, -1, 17):
            assert fn(T=T) == -2, (fn.__name__, T)
        assert fn(B=-1) == -2, fn.__name__
    assert colsum(lo=None) == -1 and colsum(act=None) == -1 and colsum(psum=None) == -1
    bad_counts = _lib.AsrConfig()
    bad_counts.num_counts = 9
    no_counts = _lib.AsrConfig()
    no_counts.gamma_margin = 1.0                # gamma_margin > 0 with no count
    for fn in (forward, backward):
        assert fn(cfg_=ctypes.byref(bad_counts)) == -2, fn.__name__
        assert fn(cfg_=ctypes.byref(no_counts)) == -2, fn.__name__
        assert fn(cfg_=None) == -1, fn.__name__
        for i in range(4):                      # log_odds, shifts, scales, psum
            assert fn(ins=(one,) * i + (None,) + (one,) * (3 - i)) == -1, (fn.__name__, i)
    # psum is required even with the count penalties off (it carries the trip count)
    plain = _lib.AsrConfig()
    assert forward(ins=(one, one, one, None), cfg_=ctypes.byref(plain)) == -1
    assert backward(ins=(one, one, one, None), cfg_=ctypes.byref(plain)) == -1
    assert "psum" in _lib.last_error()
    assert forward(outs=(None, None, one, None)) == -1         # per_image
    assert forward(outs=(one, None, None, None)) == -1         # margin
    assert forward(B=0, ins=(None, None, None, one), outs=(None, None, None, None)) == -1   # margin even at B = 0
    assert forward(B=0, ins=(None, None, None, None), outs=(None, None, one, None)) == -1   # psum even at B = 0
    assert backward(grads=(None, one)) == -1                    # g_per_image (g_margin is nullable)
    for i in range(3):
        assert backward(outs=(one,) * i + (None,) + (one,) * (2 - i)) == -1, i


def test_zero_batch_of_the_steps_entry_points(lib):
    """B = 0: the column sum and the backward are no-ops (the forward still writes margin and steps: a GPU test)"""
    assert lib.mog_asr_reg_colsum_steps(None, None, None, 0, 6, None) == 0
    cfg = _lib.AsrConfig()
    assert lib.mog_asr_reg_backward_steps(None, None, None, None, 0.0, None, None, 0, 6, ctypes.byref(cfg), None, None, None,
                                          None) == 0


def test_executed_form_refuses_cpu_tensors():
    from mog_asr_b200.asr import AsrRegulariser, asr_regularisers_executed
    reg = AsrRegulariser(canvas_size=50, max_steps=3)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        asr_regularisers_executed(reg, torch.zeros(2, 3), torch.zeros(2, 3, 2), torch.ones(2, 3), torch.ones(3, 2, dtype=torch.bool))
