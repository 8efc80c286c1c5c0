"""The training driver (``python -m mog_asr_b200.air.train``) on the CPU: its flags, the loop with the oracle's operators in
float64 fed from a step-indexed numpy source (resume bit-equality, log means), and the sharded test pass over gloo."""
import json
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from mog_asr_b200 import synth
from mog_asr_b200.air import Trainer, config_from_flags
from mog_asr_b200.air import train as T
from mog_asr_b200.air.bench_train import GlobalSeededNoise
from oracle.air_ops import OracleOps
from oracle.detection_ref import evaluation_per_instance

C3 = ["-data", "sprites", "-dn", "3", "-ds", "bbox20k", "-gb", "1", "-gs", "10", "-ga", "20"]


def numpy_source(seed):
    """``source(index, batch_size, rank, world)``: canvases of ``synth.multi_object_canvases``, each seeded by its canvas index
    (as the device feeder's stream: a function of the step index, whatever the sharding), with their counts and boxes"""
    def source(k, B, rank, world):
        first = (k * world + rank) * B
        one = [synth.multi_object_canvases(1, 50, 28, (1, 3), seed=seed * 100003 + first + b) for b in range(B)]
        canv, num = np.concatenate([c for c, _ in one]), np.concatenate([n for _, n in one])
        # ground-truth boxes for the metrics: drawn per canvas index (the generator does not return its boxes)
        boxes = np.stack([np.random.default_rng(seed * 100003 + first + b).integers(0, 30, size=(3, 4)) for b in range(B)])
        pos, size = boxes[..., :2], boxes[..., 2:] // 2 + 8
        return dict(images=torch.tensor(np.clip(canv, 0, 1).reshape(B, -1), dtype=torch.float64),
                    num=torch.tensor(num.astype(np.int32)), pos=torch.tensor(pos.astype(np.int32)),
                    size=torch.tensor(size.astype(np.int32)))
    return source


def oracle_metrics(gt_pos, gt_size, gt_num, inf_shifts, inf_scales, inf_num, cs):
    """``detection.detection_metrics`` restated by the oracle (ragged per-image lists), per-image float64 tensors"""
    P = [gt_pos[b, :int(gt_num[b])].reshape(-1).tolist() for b in range(len(gt_num))]
    S = [gt_size[b, :int(gt_num[b])].reshape(-1).tolist() for b in range(len(gt_num))]
    out = evaluation_per_instance(P, S, inf_shifts.numpy(), inf_scales.reshape(len(gt_num), -1, 1).numpy(), inf_num.numpy(), cs)
    return tuple(torch.tensor(o) for o in out)


def test_flags_map_to_config_from_flags():
    a = T.parse_args(C3)
    assert T.make_config(a, captured=False) == config_from_flags(data="sprites", dn="3", ds="bbox20k", gb=1.0, gs=10.0, ga=20.0)
    assert T.make_config(a, captured=True) == config_from_flags(data="sprites", dn="3", ds="bbox20k", gb=1.0, gs=10.0, ga=20.0,
                                                                always_max_steps=True, reference_trip_count=True)
    assert T.dataset_mode(a) == "bbox" and T.dataset_mode(T.parse_args([])) == "pixel"
    a = T.parse_args(["-dn", "13", "-gn", "1", "-gm", "100", "-gne", "10", "-zt", "0.5", "-r", "out", "-k", "c2"])
    assert T.make_config(a, False) == config_from_flags(dn="13", gn=1.0, gm=100.0, gne=10.0, zt=0.5)
    d = T.parse_args([])
    assert (d.global_batch, d.log_every, d.test_every, d.save_every, d.keep) == (64, 20, 200, 10000, 3)
    for bad in (["--unknown"], ["-x", "1"], ["-gn"], ["--steps", "0"], ["-dn13x"]):
        with pytest.raises(SystemExit):
            T.parse_args(bad)


def test_existing_results_folder_is_not_overwritten(tmp_path):
    os.makedirs(tmp_path / "run")
    (tmp_path / "run" / "log.jsonl").write_text("x\n")
    args = T.parse_args(["-r", str(tmp_path), "-k", "run", "--steps", "1"])
    with pytest.raises(SystemExit, match="exists"):
        T.train(args, "cpu", ops=OracleOps(), source=numpy_source(0), dtype=torch.float64)


def run(tmp_path, name, steps, extra=(), process_group=None):
    args = T.parse_args(["-dn", "13", "-gm", "100", "-gne", "10", "--global-batch", "4", "--steps", str(steps),
                         "--log-every", "1", "--test-every", "100", "--save-every", "1", "--keep", "2", "-r", str(tmp_path),
                         "-k", name, *extra])
    ops = OracleOps(process_group=process_group, global_batch=4)
    tr = T.train(args, "cpu", process_group=process_group, ops=ops, source=numpy_source(3), dtype=torch.float64,
                 out=open(os.devnull, "w"))
    logs = []
    if tr.rank == 0:
        with open(os.path.join(tmp_path, name, "log.jsonl")) as f:
            logs = [json.loads(l) for l in f]
        for l in logs:
            assert l.pop("images_per_sec") > 0 and l.pop("gpu") == "cpu"
    return tr, logs


def test_resume_is_bit_equal_to_the_uninterrupted_run(tmp_path):
    """float64 oracle operators on the CPU: 4 steps in one go against 2 steps + checkpoint + --resume + 2 steps.  Parameters,
    Adam's moments and step count, and every log line (less the rate) are equal bit for bit."""
    full, log_full = run(tmp_path, "full", 4)
    run(tmp_path, "split", 2)
    ck = torch.load(tmp_path / "split" / "ckpt-00000002.pt", weights_only=True)
    assert ck["step"] == 2 and ck["t"] == 2 and ck["config"]["constrains_num"] == [1, 3] and ck["flags"]["dn"] == "13"
    assert len(ck["rng"]) == len(ck["log_buffer"]) == 1
    resumed, log_res = run(tmp_path, "split", 4, ["--resume"])
    assert log_res == log_full and [l["step"] for l in log_full] == [1, 2, 3, 4]
    assert resumed.t == full.t == 4 and torch.equal(resumed.t_dev, full.t_dev)
    for a, b in zip(list(full.params) + full.m + full.v, list(resumed.params) + resumed.m + resumed.v):
        assert torch.equal(a, b)
    # a checkpoint after every step, --keep 2: the older ones are gone
    assert [os.path.basename(p) for p in T.checkpoints(tmp_path / "split")] == ["ckpt-00000003.pt", "ckpt-00000004.pt"]
    assert [os.path.basename(p) for p in T.checkpoints(tmp_path / "full")] == ["ckpt-00000003.pt", "ckpt-00000004.pt"]


def _gloo_train(rank, world, port, root, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        pg = dist.group.WORLD
        every = ["--log-every", "2"]
        full, log_full = run(root, "full", 4, every, pg)
        run(root, "split", 3, every, pg)                 # the last save, at step 3, falls inside a log interval
        res, log_res = run(root, "split", 4, every + ["--resume"], pg)
        if rank == 0:
            ret["logs"] = (log_full, log_res)
        ret[rank] = all(torch.equal(a, b) for a, b in zip(list(full.params) + full.m + full.v, list(res.params) + res.m + res.v))
        # set-up errors found on rank 0 stop every rank before training, none waits in a collective
        for key, call in (("exists", lambda: run(root, "full", 1, [], pg)),
                          ("does not split", lambda: T.train(T.parse_args(["-r", root, "-k", "odd", "--steps", "1"]), "cpu",
                                                             process_group=pg, ops=OracleOps(pg, 64), source=numpy_source(0),
                                                             dtype=torch.float64, test_size=999))):
            try:
                call()
                ret[f"{key}{rank}"] = False
            except SystemExit as e:
                ret[f"{key}{rank}"] = key in str(e)
    finally:
        dist.destroy_process_group()


def test_two_rank_resume_inside_a_log_interval_gloo(tmp_path):
    """Two gloo ranks (2 images each), logs every 2 steps: 3 steps with the last checkpoint after step 3, inside the
    interval 3-4, then --resume to step 4, against 4 steps in one go.  Every rank's log sums are part of the checkpoint,
    so the step-4 line (both ranks' shares of steps 3 and 4) is bit-equal, and so are parameters and Adam's moments."""
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ret = mp.Manager().dict()
    mp.spawn(_gloo_train, args=(2, port, str(tmp_path), ret), nprocs=2, join=True)
    log_full, log_res = ret["logs"]
    assert [l["step"] for l in log_full] == [2, 4] and [l["step"] for l in log_res] == [2, 4]
    assert log_res == log_full
    assert ret[0] and ret[1]
    assert ret["exists0"] and ret["exists1"] and ret["does not split0"] and ret["does not split1"]
    ck = torch.load(tmp_path / "split" / "ckpt-00000003.pt", weights_only=True)      # mid-interval: two different shares
    assert len(ck["rng"]) == len(ck["log_buffer"]) == 2 and not torch.equal(ck["log_buffer"][0], ck["log_buffer"][1])


def test_set_up_errors_stop_before_training(tmp_path):
    args = T.parse_args(["-r", str(tmp_path), "-k", "run", "--steps", "1", "--resume"])
    with pytest.raises(SystemExit, match="no checkpoint"):
        T.train(args, "cpu", ops=OracleOps(), source=numpy_source(0), dtype=torch.float64)


def test_logged_mean_is_the_mean_of_the_steps(tmp_path, monkeypatch):
    seen = []
    add = T.LogAccumulator.add

    def spy(self, out, batch):
        seen.append(dict(loss=float(out["loss"].detach()), elbo=float(out["elbo"].mean()), reconstruction=float(out["recon"].mean()),
                         margin=float(out["margin"]), steps=float(out["steps"]), comps=out["components"].mean(0).tolist(),
                         accuracy=float((out["rec_num_digits"] == batch["num"]).double().mean())))
        add(self, out, batch)
    monkeypatch.setattr(T.LogAccumulator, "add", spy)
    _, logs = run(tmp_path, "mean", 3, ["--log-every", "3"])
    assert len(logs) == 1 and len(seen) == 3
    got = logs[0]
    for key in ("loss", "elbo", "reconstruction", "margin", "steps", "accuracy"):
        np.testing.assert_allclose(got[key], np.mean([s[key] for s in seen]), rtol=1e-12, atol=1e-12, err_msg=key)
    for i, key in enumerate(("pr_num", "num_min", "area", "out", "size", "overlap")):
        np.testing.assert_allclose(got[key], np.mean([s["comps"][i] for s in seen]), rtol=1e-12, atol=1e-12, err_msg=key)


# ---- the test pass sharded over two gloo ranks ------------------------------------------------------------------------
TEST_N = 8


def held_out(trainer):
    noise = lambda lo, hi: (lambda kind, step, shape: GlobalSeededNoise(9, TEST_N, lo, hi, "cpu")(kind, step, shape).double())
    return T.held_out_pass(trainer, numpy_source(7), metrics=oracle_metrics, test_noise=noise, size=TEST_N)


def _gloo_worker(rank, world, port, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        cfg = config_from_flags(dn="13", gm=100.0, gne=10.0)
        tr = Trainer(cfg, "cpu", process_group=dist.group.WORLD, global_batch=TEST_N, dtype=torch.float64,
                     ops=OracleOps(process_group=dist.group.WORLD, global_batch=TEST_N))
        ret[rank] = {k: v.clone() for k, v in held_out(tr).items()}
    finally:
        dist.destroy_process_group()


def test_sharded_test_pass_equals_one_process_gloo():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ret = mp.Manager().dict()
    mp.spawn(_gloo_worker, args=(2, port, ret), nprocs=2, join=True)
    one = held_out(Trainer(config_from_flags(dn="13", gm=100.0, gne=10.0), "cpu", ops=OracleOps(), dtype=torch.float64))
    assert float(one["images"]) == TEST_N
    for r in (0, 1):
        assert float(ret[r]["images"]) == TEST_N
        assert float(ret[r]["accuracy"]) * TEST_N == float(one["accuracy"]) * TEST_N
        for k, v in one.items():
            np.testing.assert_allclose(ret[r][k].numpy(), v.numpy(), rtol=0, atol=1e-12, err_msg=k)
