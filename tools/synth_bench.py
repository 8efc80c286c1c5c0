"""Time the on-device dataset feeder: placement for every rule (``bbox``, ``disjoint``, ``pixel``) and the paste, with
square objects and with rotated objects labelled with their tight boxes.

    python tools/synth_bench.py [--reps 50] [--batch 4096]

Workloads: Multi-MNIST-like batches of 4096 canvases, 50x50 with 1-3 objects of 17-23 px (configs C2 / C4) and 64x64
with 1-3 objects of 20-25 px.  Each timed call places (or places and pastes) a fresh range of canvas indices, so
restarts and attempts vary as they do in a stream.  The rotated runs (``rot_*`` keys) draw every object's angle from
the 40 dSprites orientations (``dsprites_angles``), the full circle, so objects take up to sqrt(2) times their square.
Times are CUDA-event means after warm-up, in microseconds per batch, and the matching rates in canvases per second.
Prints one JSON line per workload, with the device name and its power limit.  Needs a CUDA device: there is no CPU path.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = [  # name, canvas, counts, size range
    ("mnist50", 50, (1, 2, 3), (17, 23)),
    ("canvas64", 64, (1, 2, 3), (20, 25)),
]
MODES = ("bbox", "disjoint", "pixel")


def power_limit_w(index):
    try:
        import pynvml
        pynvml.nvmlInit()
        return pynvml.nvmlDeviceGetPowerManagementLimit(pynvml.nvmlDeviceGetHandleByIndex(index)) / 1000.0
    except Exception:
        pass
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return float(out)
    except Exception:
        return None


def time_us(fn, reps, warmup, dev):
    import torch
    for k in range(warmup):
        fn(k)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(dev)
    e0.record()
    for k in range(reps):
        fn(warmup + k)
    e1.record()
    torch.cuda.synchronize(dev)
    return e0.elapsed_time(e1) * 1e3 / reps


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch", type=int, default=4096)
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        sys.exit("synth_bench.py needs a CUDA device (the feeder has no CPU path)")
    from mog_asr_b200 import build
    from mog_asr_b200.dataset import DeviceMultiObjectDataset, default_sprites, dsprites_angles
    build.build()
    dev = torch.device("cuda:0")
    device = dict(name=torch.cuda.get_device_name(dev), power_limit_w=power_limit_w(0),
                  sms=torch.cuda.get_device_properties(dev).multi_processor_count)
    sprites = default_sprites(256, 28, seed=0)
    B = args.batch
    for name, cs, counts, srange in WORKLOADS:
        res = dict(workload=name, canvas=cs, counts=list(counts), size_range=list(srange), batch=B, device=device)
        for mode in MODES:
            ds = DeviceMultiObjectDataset(sprites, cs, counts, srange, mode=mode, seed=5, device=dev)
            res[f"place_{mode}_us"] = round(time_us(lambda k: ds.place(k * B, B), args.reps, args.warmup, dev), 1)
            res[f"place_paste_{mode}_us"] = round(time_us(lambda k: ds.batch(k, B), args.reps, args.warmup, dev), 1)
            placed = ds.place(0, B)
            res[f"mean_objects_{mode}"] = round(float(placed[0].float().mean()), 3)
            if mode == "pixel":
                res["paste_us"] = round(time_us(lambda k: ds.paste(*placed), args.reps, args.warmup, dev), 1)
        for mode in MODES:
            ds = DeviceMultiObjectDataset(sprites, cs, counts, srange, mode=mode, seed=5, device=dev, angles=dsprites_angles())
            res[f"place_rot_{mode}_us"] = round(time_us(lambda k: ds.place(k * B, B), args.reps, args.warmup, dev), 1)
            res[f"place_paste_rot_{mode}_us"] = round(time_us(lambda k: ds.batch(k, B), args.reps, args.warmup, dev), 1)
            placed = ds.place(0, B)
            res[f"mean_objects_rot_{mode}"] = round(float(placed[0].float().mean()), 3)
            if mode == "pixel":
                res["paste_rot_us"] = round(time_us(lambda k: ds.paste(*placed), args.reps, args.warmup, dev), 1)
        for key in [k for k in res if k.startswith("place_paste_")]:
            res[key.replace("place_paste_", "canvases_per_s_").replace("_us", "")] = round(B / (res[key] * 1e-6))
        print(json.dumps(res), flush=True)
        print(f"# {name} ({B} canvases {cs}x{cs}, {device['name']}, power limit {device['power_limit_w']} W): "
              + ", ".join(f"place {m} {res[f'place_{m}_us']} us" for m in MODES) + f", paste {res['paste_us']} us; rotated: "
              + ", ".join(f"place {m} {res[f'place_rot_{m}_us']} us" for m in MODES) + f", paste {res['paste_rot_us']} us; "
              + "place + paste canvases/s: " + ", ".join(f"{m} {res[f'canvases_per_s_{m}']} / rotated {res[f'canvases_per_s_rot_{m}']}"
                                                         for m in MODES), flush=True)


if __name__ == "__main__":
    main()
