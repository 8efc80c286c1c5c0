#!/usr/bin/env python
"""Per-kernel timing of the four sampler kernels on chosen cells of the config-5 sweep (development tool).

    python tools/kbench.py --cells 256:64:prior,50:28:full --reps 5 --tag mytag

For every cell: canvas:glimpse:regime, B canvases, two theta sets; each kernel kind is timed with CUDA events on
the launch stream (inputs larger than L2) and reported in microseconds with its algorithmic bytes
(bench.py's accounting).  Writes gpurun_out/kbench_<tag>.json and prints one line per cell.
MOG_SO selects another build of the library.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--cells", default="256:64:prior")
    p.add_argument("--batch", type=int, default=16384)
    p.add_argument("--reps", type=int, default=5)
    p.add_argument("--tag", default="k")
    p.add_argument("--kinds", default="read_fwd,read_bwd,read_bwd_dtheta,write_fwd,write_bwd")
    a = p.parse_args()
    import torch
    import bench
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    peak, _ = bench.peak_hbm()
    rows = []
    for cell in a.cells.split(","):
        cs, gs, regime = cell.split(":")
        ns = argparse.Namespace(canvas=int(cs), glimpse=int(gs), regime=regime, batch=a.batch)
        bench.AIR_STEPS_SAVED = bench.AIR_STEPS
        bench.AIR_STEPS = 2
        try:
            wl = bench.GpuWorkload(ns, dev, seed=10)
            ab = wl.algorithmic_bytes()
        finally:
            bench.AIR_STEPS = bench.AIR_STEPS_SAVED
        out = {}
        for kind in a.kinds.split(","):
            for _ in range(2):
                for t in range(2):
                    wl.launch(kind, t)
            torch.cuda.synchronize(dev)
            ev = []
            for _ in range(a.reps):
                for t in range(2):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    wl.launch(kind, t)
                    e1.record()
                    ev.append((e0, e1))
            torch.cuda.synchronize(dev)
            us = float(np.median([x.elapsed_time(y) for x, y in ev])) * 1e3
            mb = ab[kind] / 1e6
            out[kind] = dict(us=us, alg_mb=mb, frac=ab[kind] / (us * 1e-6) / 1e9 / peak)
        rows.append(dict(cell=cell, batch=a.batch, kernels=out))
        print(cell, " ".join(f"{k}={v['us']:.0f}us/{v['frac']:.2f}" for k, v in out.items()), flush=True)
        del wl
        torch.cuda.empty_cache()
    os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
    with open(os.path.join(ROOT, "gpurun_out", f"kbench_{a.tag}.json"), "w") as f:
        json.dump(dict(peak=peak, rows=rows, so=os.environ.get("MOG_SO", "in-tree")), f, indent=1)


if __name__ == "__main__":
    main()
