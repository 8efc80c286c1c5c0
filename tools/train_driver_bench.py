"""python tools/train_driver_bench.py [C2 C4] [--steps N]   (single GPU)

Images/s of the training driver (``python -m mog_asr_b200.air.train``: fresh batch per step, device-side log sums, one
read per 20 steps) with the feed inside the captured step and with the feed launched eagerly before each replay, beside
``tools/train_bench.py``'s captured reference-trip-count row (4 resident batches cycled, no feed), all in one process.
The driver's rate is the mean over its log intervals after the first (the first includes the first replays).  Prints
one JSON line per row with the card's name and power limit."""
import argparse
import json
import os
import subprocess
import sys
import tempfile

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from mog_asr_b200.air import bench_train  # noqa: E402
from mog_asr_b200.air import train as driver  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, _, power = q.stdout.strip().partition(",")
    return dict(gpu=name.strip() or torch.cuda.get_device_name(0), power_limit=power.strip() or "unknown")


def driver_row(name, feed, steps, log_every=20):
    flags, gbatch = bench_train.CONFIGS[name]
    argv = []
    for k, v in flags.items():
        argv += ["-" + k, str(v)]
    with tempfile.TemporaryDirectory() as tmp:
        args = driver.parse_args(argv + ["--global-batch", str(gbatch), "--steps", str(steps), "--log-every", str(log_every),
                                         "--test-every", str(10 * steps), "--save-every", str(10 * steps),
                                         "-r", tmp, "-k", "run"])
        driver.train(args, "cuda:0", out=open(os.devnull, "w"), feed_in_graph=feed == "graph")
        with open(os.path.join(tmp, "run", "log.jsonl")) as f:
            lines = [json.loads(l) for l in f]
    rates = [l["images_per_sec"] for l in lines[1:]]
    return dict(config=name, row="driver, feed " + ("in the graph" if feed == "graph" else "eager before each replay"),
                images_per_sec=sum(rates) / len(rates), intervals=len(rates), global_batch=gbatch)


def main():
    p = argparse.ArgumentParser()
    p.add_argument("configs", nargs="*", default=["C2", "C4"])
    p.add_argument("--steps", type=int, default=120)
    p.add_argument("--repeats", type=int, default=2)
    a = p.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    info = card()
    for name in a.configs:
        for rep in range(a.repeats):          # alternate the rows: other work shares the host
            r = bench_train.run(name, dev, steps=a.steps, warmup=5, always_max_steps=True, graph=True, reference_trip_count=True)
            print(json.dumps(dict(config=name, row="train_bench captured, reference trip count (resident batches)",
                                  images_per_sec=r["images_per_sec"], repeat=rep, **info)), flush=True)
            for feed in ("graph", "eager"):
                print(json.dumps(dict(driver_row(name, feed, a.steps), repeat=rep, **info)), flush=True)


if __name__ == "__main__":
    main()
