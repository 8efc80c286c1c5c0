"""The training driver on the GPU: the device-index placement entry points under graph replay, the feed captured with the
step, resume at the first resumed step, and the sharded test pass's sums."""
import json
import os
import re
import subprocess

import numpy as np
import pytest
import torch

from mog_asr_b200 import build
from mog_asr_b200.air import Trainer, config_from_flags
from mog_asr_b200.air import train as T
from mog_asr_b200.air.bench_train import GlobalSeededNoise
from mog_asr_b200.air.evaluate import evaluate_detection_sums, sums_to_means
from mog_asr_b200.dataset import DeviceMultiObjectDataset, default_sprites, dsprites_angles

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_placement_kernels_compile_without_spills(tmp_path):
    """``-Xptxas -v`` of the placement source: the three kernels (which serve both the host-index and the ``_dev`` entry
    points) spill nothing, and the warp kernels stay within the 64 registers their 8 CTAs per SM assume"""
    flags = [f for f in build.flags() if f != "-shared"]
    res = subprocess.run([build.nvcc_path()] + flags + ["-Xptxas", "-v", "-c", os.path.join(ROOT, "mog_asr_b200", "csrc", "mog_synth.cu"),
                          "-o", str(tmp_path / "s.o")], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    text = res.stderr
    for k in ("synth_place_kernel", "synth_place_pixels_kernel", "synth_place_rotated_kernel"):
        assert k in text
    assert all(int(s) == 0 for s in re.findall(r"(\d+) bytes spill", text)), text
    regs = [int(r) for r in re.findall(r"Used (\d+) registers", text)]
    assert regs and max(regs) <= 64, text


DATASETS = {
    "box": dict(mode="disjoint"),
    "pixel": dict(mode="pixel"),
    "rotated": dict(mode="pixel", angles=dsprites_angles()),
}


@pytest.mark.parametrize("kind", sorted(DATASETS))
def test_device_index_placement_under_graph_replay(cuda_device, kind):
    """A graph captured around ``place(index_tensor, B)`` replayed at two indices gives what the host-index entry point
    gives for the same indices: num / pos / size / sprite (and theta for rotated objects), bit for bit"""
    ds = DeviceMultiObjectDataset(default_sprites(64, 28), 50, (1, 2, 3), (11, 23), seed=5, device=cuda_device, **DATASETS[kind])
    B = 300
    idx = torch.zeros((), dtype=torch.int64, device=cuda_device)
    ds.place(idx, B)                      # load the kernels before capture
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = ds.place(idx, B)
    for first in (1234, 77):
        idx.fill_(first)
        g.replay()
        ref = ds.place(first, B)
        torch.cuda.synchronize()
        assert len(out) == len(ref) == (5 if kind == "rotated" else 4)
        for a, b in zip(out, ref):
            assert torch.equal(a, b), (kind, first)
    with pytest.raises(ValueError, match="int64"):
        ds.place(idx.to(torch.int32), B)
    # a dataset on the bare "cuda" device takes an index tensor on the device that resolves to
    bare = DeviceMultiObjectDataset(default_sprites(64, 28), 50, (1, 2, 3), (11, 23), seed=5, device="cuda", **DATASETS[kind])
    with torch.cuda.device(cuda_device):
        got = bare.place(idx, 8)
    assert torch.equal(got[0], ds.place(77, 8)[0])


C2 = dict(data="mnist", dn="13", gm=100.0, gne=10.0)


@pytest.mark.parametrize("in_graph", [True, False], ids=["graph_feed", "eager_feed"])
def test_captured_feed_trains_on_the_dataset_batches(cuda_device, in_graph):
    """The captured step with the feed: before replay k the step's input buffer holds ``clamp(dataset.batch(k, B))``
    bit for bit, counts included, and the device index reads k"""
    cfg = config_from_flags(always_max_steps=True, reference_trip_count=True, **C2)
    ds = DeviceMultiObjectDataset(default_sprites(), 50, (1, 3), (17, 23), mode="pixel", seed=3, device=cuda_device)
    B = 16
    tr = Trainer(cfg, cuda_device, global_batch=B).capture(B, feed=T.make_feed(ds, B, 0, 1), feed_in_graph=in_graph)
    tr.start_feed(7)
    for k in range(7, 10):
        if in_graph:
            ref = ds.batch(k, B)
            torch.cuda.synchronize()
            assert torch.equal(tr.static_images, torch.clamp(ref["images"], 0.0, 1.0)), k
            assert torch.equal(tr.static_batch["num"], ref["num"]) and int(tr.feed_step) == k
        out = tr.step_graph()
        if not in_graph:
            ref = ds.batch(k, B)
            torch.cuda.synchronize()
            assert torch.equal(tr.static_images, torch.clamp(ref["images"], 0.0, 1.0)), k
        assert torch.isfinite(out["loss"]).item()


def run_driver(root, name, steps, extra=()):
    args = T.parse_args(["-dn", "13", "-gm", "100", "-gne", "10", "--global-batch", "32", "--steps", str(steps), "--log-every", "1",
                         "--test-every", "2", "--save-every", "1", "--keep", "10", "-r", str(root), "-k", name, *extra])
    tr = T.train(args, "cuda:0", out=open(os.devnull, "w"), test_size=200)
    with open(os.path.join(root, name, "log.jsonl")) as f:
        return tr, [json.loads(l) for l in f]


def head_second_layers(model):
    """names of the (mean, log-variance) heads' second-layer weights and biases: their gradients are the atomically
    summed ones (csrc/mog_air_head.cu)"""
    from mog_asr_b200.air.model import _MeanVar
    return {f"{n}.{br}.{w}" for n, mod in model.named_modules() if isinstance(mod, _MeanVar) for br in ("m", "v")
            for w in ("weight", "bias")}


def test_resume_reproduces_the_first_resumed_step(cuda_device, tmp_path):
    """Run 3 steps, with a held-out pass (200 canvases) after step 2 and a checkpoint after each step; resume a copy of the
    step-2 checkpoint and run step 3 again.

    The loss and every logged variable of step 3 equal the uninterrupted run's bit for bit: same parameters, Adam state,
    batch and noise (the default CUDA generator's offset, advanced by the graph and by the held-out pass, is restored
    after capture), and with 32 images the forward's one atomic sum (asr_colsum) adds one warp's value to zeros.

    In the step's backward the only atomic sums are those of the heads' second-layer weight and bias gradients.  Clipping
    is per variable, so every other parameter and both its Adam moments must be bit-equal to the uninterrupted run's
    step-3 checkpoint.  For the head tensors, each gradient entry is a sum of at most N = 30 per-CTA partials (B * T / 8
    rows' CTAs plus one call per step) added in any order: two orders differ by at most 2 N u sum|partial|, u = 2^-24.  The
    partials are not observable here, so sum|partial| is taken as 16 times the tensor's largest gradient entry (the
    gradient comes from the uninterrupted run's moments, g = (m3 - b1 m2) / (1 - b1)).  That bounds |dm| by (1 - b1) dg and
    |dv| by (1 - b2)(2 |g| dg + dg^2); the parameters may then differ by the first-order change of Adam's update."""
    full, log_full = run_driver(tmp_path, "full", 3)
    with open(tmp_path / "full" / "test.jsonl") as f:
        tests = [json.loads(l) for l in f]
    assert [t["step"] for t in tests] == [2] and tests[0]["images"] == 200 and len(tests[0]["precision"]) == 11
    os.makedirs(tmp_path / "res")
    src = tmp_path / "full" / "ckpt-00000002.pt"
    (tmp_path / "res" / src.name).write_bytes(src.read_bytes())
    res, log_res = run_driver(tmp_path, "res", 3, ["--resume"])
    assert [l["step"] for l in log_res] == [3]
    a, b = dict(log_full[2]), dict(log_res[0])
    for d in (a, b):
        d.pop("images_per_sec")
    assert a == b
    assert res.t == full.t == 3 and torch.equal(res.t_dev, full.t_dev)

    b1, b2, eps, u = 0.9, 0.999, 1e-8, 2.0 ** -24
    lr_t = full.cfg.learning_rate * np.sqrt(1 - b2 ** 3) / (1 - b1 ** 3)
    ck2 = torch.load(tmp_path / "full" / "ckpt-00000002.pt", weights_only=True, map_location=cuda_device)
    ck3 = torch.load(tmp_path / "full" / "ckpt-00000003.pt", weights_only=True, map_location=cuda_device)
    heads = head_second_layers(res.model)
    names = [n for n, _ in res.model.named_parameters()]
    assert len(heads) == 12 and heads <= set(names)
    ulp = lambda x: torch.finfo(torch.float32).eps * x.abs()
    for i, name in enumerate(names):
        p, m, v = res.model.state_dict()[name], res.m[i], res.v[i]
        p3, m3, v3 = ck3["model"][name], ck3["adam_m"][i], ck3["adam_v"][i]
        if name not in heads:
            assert torch.equal(p, p3) and torch.equal(m, m3) and torch.equal(v, v3), name
            continue
        g = (m3.double() - b1 * ck2["adam_m"][i].double()) / (1 - b1)
        dg = 2 * 30 * u * 16 * float(g.abs().max())
        dm, dv = (m - m3).double().abs(), (v - v3).double().abs()
        assert bool((dm <= (1 - b1) * dg + 2 * ulp(m3)).all()), name
        assert bool((dv <= (1 - b2) * (2 * g.abs() * dg + dg * dg) + 2 * ulp(v3)).all()), name
        sv = v3.double().sqrt()
        dp = lr_t * (dm / (sv + eps) + m3.double().abs() * dv / (2 * sv.clamp(min=1e-30) * (sv + eps) ** 2))
        assert bool(((p - p3).double().abs() <= 2 * dp + 4 * ulp(p3)).all()), name


class Replayed:
    """the test model's outputs for a whole set, served row range by row range (``rows``) as ``evaluate_detection_sums``
    asks for them: the shards then score exactly the per-image values the whole set scores"""

    def __init__(self, model, out):
        self.cfg, self.out, self.rows = model.cfg, out, slice(None)

    def __call__(self, images, **kw):
        return {k: self.out[k][self.rows] for k in ("rec_shifts", "rec_scales", "rec_num_digits")}


def test_two_shards_of_the_test_set_sum_to_the_whole(cuda_device):
    """``evaluate_detection_sums`` of two halves of the held-out set, added, against the whole set.  On the same per-image
    model outputs: image and correct counts exactly, the means to 1e-12 (only the order of float64 sums differs).  Through
    the fp32 model itself, with the same per-image noise: counts exactly; the means within 1e-6, because the library GEMMs
    pick different tilings for 100 rows than for 200 and the boxes then differ in their last bits."""
    cfg = config_from_flags(always_max_steps=True, reference_trip_count=True, **C2)
    ds = DeviceMultiObjectDataset(default_sprites(), 50, (1, 3), (17, 23), mode="pixel", seed=T.TEST_SEED, device=cuda_device)
    tr = Trainer(cfg, cuda_device, global_batch=64)
    N, H = 200, 100
    noise = lambda lo, hi: GlobalSeededNoise(4, N, lo, hi, cuda_device)
    whole_batch = ds.batch(0, N)
    whole = evaluate_detection_sums(tr.model, whole_batch, noise=noise(0, N))
    with torch.no_grad():
        rep = Replayed(tr.model, tr.model(torch.clamp(whole_batch["images"], 0.0, 1.0), noise=noise(0, N), train=False))
    exact = 0
    for r in (0, 1):
        rep.rows = slice(r * H, (r + 1) * H)
        exact = exact + evaluate_detection_sums(rep, ds.batch(0, H, r, 2))
    parts = sum(evaluate_detection_sums(tr.model, ds.batch(0, H, r, 2), noise=noise(r * H, (r + 1) * H)) for r in (0, 1))
    mw = sums_to_means(whole.cpu())
    for got, tol in ((exact, 1e-12), (parts, 1e-6)):
        assert float(got[-1]) == N and float(got[-2]) == float(whole[-2])
        mg = sums_to_means(got.cpu())
        for k in mw:
            np.testing.assert_allclose(mg[k].numpy(), mw[k].numpy(), rtol=0, atol=tol, err_msg=k)
