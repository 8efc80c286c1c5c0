#!/usr/bin/env python
"""bench.py -- STN glimpses/sec (forward+backward) on the BASELINE config-5 workload, one JSON line.

    python bench.py --gpus N --steps K --warmup W            # this repo's sm_100a kernels
    python bench.py --impl reference --steps K --warmup W    # the reference path's CPU restatement
    python bench.py --steps K --warmup W --dump-outputs DIR  # also write the last timed step's outputs (a sample) to DIR

Workload (SURVEY 8(d), BASELINE.json configs[4]): the LARGEST cell of the config-5 sweep -- canvas 256x256,
glimpse 64x64, prior-like theta (`--canvas/--glimpse/--regime` select any other cell, `--sweep` runs them
all; the reference's own Multi-MNIST shapes are `--canvas 50 --glimpse 28`).  Per GPU B = 16384 canvases (C = 1),
8 sequential AIR steps with a distinct theta per step; every step does what an AIR step asks of the
sampler -- a *read* glimpse (canvas -> glimpse, theta_r) and a *write* glimpse (glimpse -> canvas,
theta_w), each forward + backward(dU + dtheta).  One bench "step" = those 8 AIR steps over the batch
= 16 * B glimpses.  Batch shards are independent, so N GPUs run N shards (weak scaling, no collective).

`value`: glimpses/s with inputs resident in HBM (CUDA events, max over ranks).
`e2e`  : the same 16*B glimpses through the host-buffer entry points (pinned host arrays in, host arrays out,
         copies inside the timed region): mog_stn_batch_fwd_bwd_host for the reads, mog_stn_write_composite_host for
         the writes (the AIR loop's data flow); `e2e.separate_write_canvases` = every write step's canvas on its own.
`roofline`: algorithmic bytes (SURVEY 8(d): fwd 4(F+O)+24, bwd 4(O+F+S)+48 per glimpse, F = distinct
         source pixels addressed) of the dominant kernel / its mean duration, vs MEASURED_PEAKS.json.
`cpu_baseline`: oracle C restatement (all host threads) on a bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "stn_glimpses_per_sec_fwd_bwd"
UNIT = "glimpses/s"
AIR_STEPS = 8


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=20)
    p.add_argument("--warmup", type=int, default=5)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--canvas", type=int, default=256)
    p.add_argument("--glimpse", type=int, default=64)
    p.add_argument("--batch", type=int, default=16384, help="canvases per GPU")
    p.add_argument("--regime", default="prior", choices=["prior", "full"])
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--no-cpu", action="store_true")
    p.add_argument("--no-train", action="store_true", help="skip the AIR-ASR training-step section")
    p.add_argument("--cpu-sample", type=int, default=0, help="canvases in the CPU-baseline sample (0 = sized for ~1 s per step)")
    p.add_argument("--e2e-batch", type=int, default=0, help="canvases per GPU in the end-to-end leg (0 = the full batch)")
    p.add_argument("--sweep", action="store_true", help="run the whole config-5 sweep, write profiles/sweep_*.json")
    p.add_argument("--tag", default="", help="suffix for files written under profiles/")
    p.add_argument("--dump-outputs", metavar="DIR", default="",
                   help="after the timed steps, write the last step's outputs (a fixed sample of the batch) as DIR/<name>.npy")
    a = p.parse_args()
    if a.dump_outputs and (a.impl == "reference" or a.sweep):
        p.error("--dump-outputs records the GPU arm's headline workload: not with --impl reference or --sweep")
    return a


def workload_name(a):
    return (f"C5 STN sweep cell: canvas {a.canvas}x{a.canvas} <-> glimpse {a.glimpse}x{a.glimpse}, {AIR_STEPS} AIR steps "
            f"(read+write, fwd+bwd dU+dtheta), batch {a.batch}/GPU, theta={a.regime}-like")


def config_dict(a):
    """`config` of the JSON line: identical for both arms (what differs between them lives in `cpu_baseline.sample`)."""
    ws_mb = a.batch * (2 * a.canvas ** 2 + 2 * a.glimpse ** 2) * 4 / 1e6
    return dict(workload=workload_name(a),
                l2=f"inputs larger than L2 (per-call working set {ws_mb:.0f} MB vs 126 MB L2); no flush",
                timing="GPU arm: CUDA events on the launch stream, max over ranks; CPU arm: wall clock around the same calls")


CPU_THREADS_CAP = 16   # the CPU arm runs on min(16, usable host threads): the ratio should not move with the host's core count


def peak_hbm():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


# --------------------------------------------------------------------------------------------------
# CPU legs: the oracle's C restatement, all host threads, bounded sample of the same workload
# --------------------------------------------------------------------------------------------------
def cpu_workload(a, nsample):
    from mog_asr_b200 import synth
    rng = np.random.default_rng(10)
    U = rng.random((nsample, a.canvas, a.canvas, 1), dtype=np.float32)
    W = rng.random((nsample, a.glimpse, a.glimpse, 1), dtype=np.float32)
    gen = synth.sxy_prior_like if a.regime == "prior" else synth.sxy_full_cover
    th_r, th_w = [], []
    for t in range(AIR_STEPS):
        s, x, y = gen(nsample, seed=100 + t)
        th_r.append(synth.theta_read(s, x, y))
        th_w.append(synth.theta_write(s, x, y))
    g_r = rng.normal(size=(nsample, a.glimpse, a.glimpse, 1)).astype(np.float32)
    g_w = rng.normal(size=(nsample, a.canvas, a.canvas, 1)).astype(np.float32)
    return U, W, th_r, th_w, g_r, g_w


def host_threads():
    """Host threads this process may use (torchrun exports OMP_NUM_THREADS=1, which is not what we want)."""
    return len(os.sched_getaffinity(0))


def cpu_threads():
    return min(CPU_THREADS_CAP, host_threads())


def cpu_step(a, wl, nthreads=0):
    from oracle import stn_ref_c as RC
    U, W, th_r, th_w, g_r, g_w = wl
    for t in range(AIR_STEPS):
        RC.forward(U, th_r[t], (a.glimpse, a.glimpse), nthreads=nthreads)
        RC.backward(U, th_r[t], (a.glimpse, a.glimpse), g_r, nthreads=nthreads)
        RC.forward(W, th_w[t], (a.canvas, a.canvas), nthreads=nthreads)
        RC.backward(W, th_w[t], (a.canvas, a.canvas), g_w, nthreads=nthreads)


def cpu_measure(a, steps, warmup, nsample, one_thread_too=True):
    """The oracle's C restatement of the reference sampler on `cpu_threads()` host threads (capped so that the figure does
    not move with the host), on a bounded sample of the same workload; beside it the single-thread figure -- the
    reference's own setting (train_air_pr.py:243-244: intra_op = inter_op = 1)."""
    wl = cpu_workload(a, nsample)
    cores = cpu_threads()
    for _ in range(warmup):
        cpu_step(a, wl, cores)
    t0 = time.perf_counter()
    for _ in range(steps):
        cpu_step(a, wl, cores)
    dt = time.perf_counter() - t0
    val = nsample * 2 * AIR_STEPS * steps / dt
    out = dict(value=val, unit=UNIT, cores=cores, kind="port",
               sample=f"{nsample} canvases x {AIR_STEPS} AIR steps x (read+write) fwd+bwd x {steps} steps, "
                      f"oracle/stn_ref.c with OpenMP over images ({cores} threads = min({CPU_THREADS_CAP}, usable); "
                      f"os.cpu_count()={os.cpu_count()}, affinity={host_threads()}); the reference is TF-1.12 Python, not "
                      f"installable here -- its sampler restated in C")
    if one_thread_too:
        n1 = max(8, nsample // 8)
        wl1 = cpu_workload(a, n1)
        cpu_step(a, wl1, 1)
        t0 = time.perf_counter()
        cpu_step(a, wl1, 1)
        out["value_1thread"] = n1 * 2 * AIR_STEPS / (time.perf_counter() - t0)
        out["sample_1thread"] = f"{n1} canvases, 1 step, 1 thread (the reference trainer's own thread setting)"
    return out, dt / steps * 1e3


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cb, ms = cpu_measure(a, a.steps, a.warmup, a.cpu_sample)
    line = dict(impl="reference", metric=METRIC, value=cb["value"], unit=UNIT, n_gpus=a.gpus, steps=a.steps,
                warmup=a.warmup, ms_per_step=ms, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32",
                data="synthetic", config=config_dict(a),
                cpu_baseline=cb, e2e=dict(value=cb["value"], unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                gpu_launches=0)
    emit(line)


# --------------------------------------------------------------------------------------------------
# clocks
# --------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    BAD = {"hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40, "hw_power_brake": 0x80}
    INFO = {"sw_power_cap": 0x4, "gpu_idle": 0x1, "applications_clocks_setting": 0x2, "sync_boost": 0x10}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag, self.ok = index, [], False, False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        while not self.stop_flag:
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    reasons = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.samples.append((time.perf_counter(), sm, reasons))
            except Exception:
                pass
            time.sleep(0.01)

    def summary(self, t0, t1):
        if not self.ok:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvml unavailable"])
        sel = [s for s in self.samples if t0 <= s[0] <= t1] or self.samples[-3:]
        mx = self.nv.nvmlDeviceGetMaxClockInfo(self.h, self.nv.NVML_CLOCK_SM)
        bits = 0
        for s in sel:
            bits |= s[2]
        names = [k for k, v in {**self.BAD, **self.INFO}.items() if bits & v and k != "gpu_idle"]
        return dict(sm_mhz=float(np.median([s[1] for s in sel])) if sel else None, sm_max_mhz=float(mx),
                    reasons=names, samples=len(sel))


# --------------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------------
def footprint_counts(torch, M, theta, in_size, out_size):
    """(F[b], G[b]): F = distinct source pixels image b addresses, G = output pixels whose taps are inside the source on
    both axes (the only part of the upstream gradient that reaches dU or dtheta: outside it the taps cancel).  For the
    axis-aligned thetas of this workload both are cross products of per-axis counts."""
    Hs, Ws = in_size
    Ho, Wo = out_size
    B = theta.shape[0]
    F = torch.empty(B, dtype=torch.int64, device=theta.device)
    G = torch.empty(B, dtype=torch.int64, device=theta.device)
    step = max(1, (1 << 27) // (Ho * Wo))
    for b0 in range(0, B, step):
        c = M.stn_corners(theta[b0:b0 + step], in_size, out_size).view(4, -1, Ho, Wo).long()
        nb = c.shape[1]
        xs = torch.zeros((nb, Ws), dtype=torch.bool, device=theta.device)
        xs.scatter_(1, c[0, :, 0, :], True)
        xs.scatter_(1, c[1, :, 0, :], True)
        ys = torch.zeros((nb, Hs), dtype=torch.bool, device=theta.device)
        ys.scatter_(1, c[2, :, :, 0], True)
        ys.scatter_(1, c[3, :, :, 0], True)
        F[b0:b0 + nb] = xs.sum(1) * ys.sum(1)
        G[b0:b0 + nb] = (c[0, :, 0, :] != c[1, :, 0, :]).sum(1) * (c[2, :, :, 0] != c[3, :, :, 0]).sum(1)
    return F, G


class GpuWorkload:
    def __init__(self, a, dev, seed):
        import torch
        import mog_asr_b200 as M
        from mog_asr_b200 import _lib, synth
        self.torch, self.M, self.L, self.lib = torch, M, _lib.load(), _lib
        self.a, self.dev = a, dev
        B, cs, gs = a.batch, a.canvas, a.glimpse
        g = torch.Generator(device=dev).manual_seed(seed)
        self.U = torch.rand((B, cs, cs, 1), device=dev, generator=g)                  # canvases (read source)
        self.W = torch.rand((AIR_STEPS, B, gs, gs, 1), device=dev, generator=g)       # per-step windows (write source)
        gen = synth.sxy_prior_like if a.regime == "prior" else synth.sxy_full_cover
        thr, thw = [], []
        for t in range(AIR_STEPS):
            s, x, y = gen(B, seed=seed * 1000 + 100 + t)
            thr.append(synth.theta_read(s, x, y))
            thw.append(synth.theta_write(s, x, y))
        self.th_r = torch.tensor(np.stack(thr), device=dev)
        self.th_w = torch.tensor(np.stack(thw), device=dev)
        self.g_r = torch.randn((AIR_STEPS, B, gs, gs, 1), device=dev, generator=g)
        self.g_w = torch.randn((AIR_STEPS, B, cs, cs, 1), device=dev, generator=g)
        self.out_r = torch.empty((B, gs, gs, 1), device=dev)
        self.out_w = torch.empty((B, cs, cs, 1), device=dev)
        self.dU_r = torch.empty((B, cs, cs, 1), device=dev)
        self.dU_w = torch.empty((B, gs, gs, 1), device=dev)
        self.dth_r = torch.empty((B, 6), device=dev)
        self.dth_w = torch.empty((B, 6), device=dev)
        self.stream = torch.cuda.current_stream(dev).cuda_stream
        self.kinds = ("read_fwd", "read_bwd", "write_fwd", "write_bwd")
        self.nsteps = AIR_STEPS

    def launch(self, kind, t):
        a, L, ck = self.a, self.L, self.lib.check
        B, cs, gs, st = a.batch, a.canvas, a.glimpse, self.stream
        if kind == "read_fwd":
            ck(L.mog_stn_forward(self.U.data_ptr(), self.th_r[t].data_ptr(), self.out_r.data_ptr(), B, cs, cs, 1, gs, gs, 1, st), kind)
        elif kind == "read_bwd":
            ck(L.mog_stn_backward(self.U.data_ptr(), self.th_r[t].data_ptr(), self.g_r[t].data_ptr(), self.dU_r.data_ptr(),
                                  self.dth_r.data_ptr(), B, cs, cs, 1, gs, gs, 1, st), kind)
        elif kind == "read_bwd_dtheta":   # the AIR read call site: the input batch needs no gradient (dU = NULL)
            ck(L.mog_stn_backward(self.U.data_ptr(), self.th_r[t].data_ptr(), self.g_r[t].data_ptr(), None,
                                  self.dth_r.data_ptr(), B, cs, cs, 1, gs, gs, 1, st), kind)
        elif kind == "write_fwd":
            ck(L.mog_stn_forward(self.W[t].data_ptr(), self.th_w[t].data_ptr(), self.out_w.data_ptr(), B, gs, gs, 1, cs, cs, 1, st), kind)
        else:
            ck(L.mog_stn_backward(self.W[t].data_ptr(), self.th_w[t].data_ptr(), self.g_w[t].data_ptr(), self.dU_w.data_ptr(),
                                  self.dth_w.data_ptr(), B, gs, gs, 1, cs, cs, 1, st), kind)

    def step(self, events=None):
        torch = self.torch
        for t in range(AIR_STEPS):
            for kind in self.kinds:
                if events is not None:
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    self.launch(kind, t)
                    e1.record()
                    events[kind].append((e0, e1))
                else:
                    self.launch(kind, t)

    def algorithmic_bytes(self):
        """Mean algorithmic bytes per launch for each kernel kind.  SURVEY 8(d) with one correction (VERDICT r1, weak #2):
        a backward is charged only the part G of the upstream gradient whose taps lie inside the source -- the rest
        cancels exactly and no implementation needs to read it -- instead of the whole output O:
        fwd 4(F+O)+24, bwd(dU+dtheta) 4(G+F+S)+48, bwd(dtheta only) 4(G+F)+48.  `survey` keeps the uncorrected figures."""
        torch, a = self.torch, self.a
        cs, gs = a.canvas, a.glimpse
        n = self.th_r.shape[0]
        out = {k: 0.0 for k in ("read_fwd", "read_bwd", "read_bwd_dtheta", "write_fwd", "write_bwd")}
        self.survey_bytes = {k: 0.0 for k in ("read_bwd", "write_bwd")}
        for t in range(n):
            Fr, Gr = (v.double() for v in footprint_counts(torch, self.M, self.th_r[t], (cs, cs), (gs, gs)))
            Fw, Gw = (v.double() for v in footprint_counts(torch, self.M, self.th_w[t], (gs, gs), (cs, cs)))
            O_r, S_r, O_w, S_w = gs * gs, cs * cs, cs * cs, gs * gs
            out["read_fwd"] += float((4 * (Fr + O_r) + 24).sum()) / n
            out["read_bwd"] += float((4 * (Gr + Fr + S_r) + 48).sum()) / n
            out["read_bwd_dtheta"] += float((4 * (Gr + Fr) + 48).sum()) / n
            out["write_fwd"] += float((4 * (Fw + O_w) + 24).sum()) / n
            out["write_bwd"] += float((4 * (Gw + Fw + S_w) + 48).sum()) / n
            self.survey_bytes["read_bwd"] += float((4 * (O_r + Fr + S_r) + 48).sum()) / n
            self.survey_bytes["write_bwd"] += float((4 * (O_w + Fw + S_w) + 48).sum()) / n
        return out


DUMP_BYTES = 32 << 20   # --dump-outputs: data bytes written in all


def dump_outputs(wl, out_dir):
    """What the timed step hands back after its last AIR step -- the read glimpse with dU and dtheta, the written canvas with
    dW and dtheta -- for a fixed, seeded sample of the batch (as many images as fit DUMP_BYTES), as float32 .npy files.
    The inputs are seeded too, so two builds run with the same arguments can be compared output for output."""
    torch, a = wl.torch, wl.a
    outputs = dict(read_out=wl.out_r, read_dU=wl.dU_r, read_dtheta=wl.dth_r,
                   write_out=wl.out_w, write_dU=wl.dU_w, write_dtheta=wl.dth_w)
    per_image = sum(t[0].numel() * t.element_size() for t in outputs.values())
    n = min(a.batch, DUMP_BYTES // per_image)
    if n == 0:
        raise SystemExit(f"--dump-outputs: one image's outputs ({per_image} bytes) exceed {DUMP_BYTES} bytes")
    idx = torch.from_numpy(np.sort(np.random.default_rng(0).choice(a.batch, n, replace=False))).to(wl.dev)
    os.makedirs(out_dir, exist_ok=True)
    for name, t in outputs.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.index_select(0, idx).cpu().numpy())


def e2e_measure(a, dev, steps, warmup, composite=True):
    """Same 16*B glimpses per step, host (pinned) arrays in and out through the host entry points.  Read direction: ONE
    mog_stn_batch_fwd_bwd_host call (the reference's batch_transformer form: the canvases cross the bus once for their 8
    thetas, dU -- summed over the 8 steps, what autodiff of 8 reads of one canvas yields -- comes back once).  Write
    direction, composite=True (the AIR loop's data flow, :592-600 + :718-727): ONE mog_stn_write_composite_host call -- 8
    distinct windows per image written onto one canvas per image, the canvas gradient differentiated back to all 8 steps
    (dW, dtheta, dz); composite=False: 8 mog_stn_fwd_bwd_host calls, every step with its own output canvas and gradient
    (the device-resident leg's form; 8x the canvas traffic)."""
    import torch
    from mog_asr_b200 import synth
    from mog_asr_b200.host_api import HostCompositeWriter, HostSampler
    B, cs, gs, T = a.e2e_batch, a.canvas, a.glimpse, AIR_STEPS
    pin = lambda *shape: torch.empty(shape, dtype=torch.float32).pin_memory()
    gdev = torch.Generator(device=dev).manual_seed(10)   # fill the host arrays from device-generated data (fast)

    def filled(t, normal):
        flat = t.view(-1)
        for o in range(0, flat.numel(), 1 << 28):
            n = min(1 << 28, flat.numel() - o)
            flat[o:o + n].copy_((torch.randn if normal else torch.rand)((n,), device=dev, generator=gdev))
        return t
    U_h, g_r = filled(pin(B, cs, cs, 1), False), filled(pin(B, T, gs, gs, 1), True)
    gen = synth.sxy_prior_like if a.regime == "prior" else synth.sxy_full_cover
    th_r, th_w = [], []
    for t in range(T):
        s, x, y = gen(B, seed=100 + t)
        th_r.append(synth.theta_read(s, x, y))
        th_w.append(synth.theta_write(s, x, y))
    th_r = torch.from_numpy(np.ascontiguousarray(np.stack(th_r, 1))).pin_memory()          # [B, T, 6]
    out_r, dU_r, dth_r = pin(B * T, gs, gs, 1), pin(B, cs, cs, 1), pin(B, T, 6)
    chunk = max(256, min(512, B // 8))
    rd = HostSampler(dev, (cs, cs), (gs, gs), 1, chunk=max(32, chunk // 4), transforms=T)   # measured: tools/e2e_probe.py
    fl = 4
    h2d = fl * (U_h.numel() + g_r.numel() + th_r.numel())
    d2h = fl * (out_r.numel() + dU_r.numel() + dth_r.numel())
    launches = 2 * (-(-B // rd.chunk))                                   # forward + backward per chunk
    if composite:
        W_h, g_c = filled(pin(T, B, gs, gs), False), filled(pin(B, cs, cs), True)
        z_h = filled(pin(T, B), False)
        th_wh = torch.from_numpy(np.ascontiguousarray(np.stack(th_w, 0))).pin_memory()     # [T, B, 6]
        canvas, dW, dth_w, dz = pin(B, cs, cs), pin(T, B, gs, gs), pin(T, B, 6), pin(T, B)
        wr = HostCompositeWriter(dev, (gs, gs), (cs, cs), steps=T, chunk=chunk, nstreams=4)

        def write():
            wr.fwd_bwd(W_h, th_wh, z_h, g_c, canvas=canvas, dW=dW, dtheta=dth_w, dz=dz)
        h2d += fl * (W_h.numel() + th_wh.numel() + z_h.numel() + g_c.numel())
        d2h += fl * (canvas.numel() + dW.numel() + dth_w.numel() + dz.numel())
        launches += 2 * T * (-(-B // wr.chunk))
        api = ("read: mog_stn_batch_fwd_bwd_host (canvases uploaded once for the 8 thetas, dU summed over them, downloaded once); "
               "write: mog_stn_write_composite_host (8 distinct windows per image composited onto one canvas per image, the canvas "
               "gradient differentiated back to the 8 windows / thetas / z_pres: the AIR loop's data flow); pinned host arrays "
               "in/out, chunked over 3-4 streams")
    else:
        W_h, g_w = filled(pin(B, gs, gs, 1), False), filled(pin(B, cs, cs, 1), True)
        th_wl = [torch.from_numpy(t).pin_memory() for t in th_w]
        out_w, dU_w, dth_w = pin(B, cs, cs, 1), pin(B, gs, gs, 1), pin(B, 6)
        wr = HostSampler(dev, (gs, gs), (cs, cs), 1, chunk=chunk)

        def write():
            for t in range(T):
                wr.fwd_bwd(W_h, th_wl[t], g_w, out=out_w, dU=dU_w, dtheta=dth_w)
        h2d += fl * T * (W_h.numel() + g_w.numel() + 6 * B)
        d2h += fl * T * (out_w.numel() + dU_w.numel() + 6 * B)
        launches += T * 2 * (-(-B // wr.chunk))
        api = ("read: mog_stn_batch_fwd_bwd_host; write: 8 x mog_stn_fwd_bwd_host (every step its own 256x256 output canvas and "
               "upstream gradient across the bus); pinned host arrays in/out, chunked over 3 streams")

    def step():
        rd.batch_fwd_bwd(U_h, th_r, g_r, out=out_r, dU=dU_r, dtheta=dth_r)
        write()

    for _ in range(warmup):
        step()
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    torch.cuda.synchronize(dev)
    dt = (time.perf_counter() - t0) / steps
    return dt, h2d, d2h, launches, api


def config1_section(dev, no_cpu):
    """BASELINE configs[0]: glimpse read 50x50 -> 28x28, 3 steps, batch 64 (launch-bound: time, not roofline)."""
    import torch
    import mog_asr_b200 as M
    from mog_asr_b200 import _lib, synth
    L = _lib.load()
    B, cs, gs, T = 64, 50, 28, 3
    canv, _ = synth.multi_object_canvases(B, cs, 28, (1, 2, 3), seed=0)
    U = torch.tensor(canv[..., None], device=dev)
    ths = [torch.tensor(synth.theta_read(*synth.sxy_prior_like(B, seed=1 + t)), device=dev) for t in range(T)]
    g = torch.randn((B, gs, gs, 1), device=dev)
    out, dU, dth = torch.empty((B, gs, gs, 1), device=dev), torch.empty_like(U), torch.empty((B, 6), device=dev)
    def step():
        st = torch.cuda.current_stream(dev).cuda_stream   # (the capture below runs on its own stream)
        for t in range(T):
            _lib.check(L.mog_stn_forward(U.data_ptr(), ths[t].data_ptr(), out.data_ptr(), B, cs, cs, 1, gs, gs, 1, st), "fwd")
            _lib.check(L.mog_stn_backward(U.data_ptr(), ths[t].data_ptr(), g.data_ptr(), dU.data_ptr(), dth.data_ptr(),
                                          B, cs, cs, 1, gs, gs, 1, st), "bwd")
    for _ in range(20):
        step()
    reps = 200
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(dev)
    e0.record()
    for _ in range(reps):
        step()
    e1.record()
    torch.cuda.synchronize(dev)
    us = e0.elapsed_time(e1) * 1e3 / reps
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        step()
    for _ in range(20):
        graph.replay()
    torch.cuda.synchronize(dev)
    e0.record()
    for _ in range(reps):
        graph.replay()
    e1.record()
    torch.cuda.synchronize(dev)
    us_graph = e0.elapsed_time(e1) * 1e3 / reps
    res = dict(workload="C1: read 50x50->28x28, 3 steps, batch 64, fwd+bwd(dU+dtheta), 6 launches",
               gpu_us_eager=us, gpu_us_graph=us_graph, glimpses_per_sec_eager=B * T / (us * 1e-6),
               glimpses_per_sec_graph=B * T / (us_graph * 1e-6))
    if not no_cpu:
        from oracle import stn_ref_c as RC
        Un, gn = U.cpu().numpy(), g.cpu().numpy()
        thn = [t.cpu().numpy() for t in ths]
        for nthreads, key in ((1, "cpu_us_1thread"), (host_threads(), "cpu_us_all_threads")):
            for _ in range(3):
                RC.forward(Un, thn[0], (gs, gs), nthreads=nthreads)
            t0 = time.perf_counter()
            n = 20
            for _ in range(n):
                for t in range(T):
                    RC.forward(Un, thn[t], (gs, gs), nthreads=nthreads)
                    RC.backward(Un, thn[t], (gs, gs), gn, nthreads=nthreads)
            res[key] = (time.perf_counter() - t0) / n * 1e6
        res["cpu_cores"] = host_threads()
    return res


def aux_section(dev):
    """The small kernels around the sampler: fused ASR regularisers (latency-bound: us per call, config 3 shape) and
    the fused reconstruction loss (HBM-bound: GB/s over 8 B/pixel forward, 12 B/pixel backward)."""
    import torch
    import mog_asr_b200 as M
    from mog_asr_b200.air import config_from_flags, CudaOps
    peak, _ = peak_hbm()

    def timeit(fn, reps):
        for _ in range(5):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(dev)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1) * 1e3 / reps   # us

    out = {}
    # ASR regularisers, config 3: B = 256, T = 6, -dn 3 -gb 1 -gs 10 -ga 20 (forward + backward, 2 launches)
    cfg = config_from_flags("sprites", "3", ds="bbox20k", gb=1.0, gs=10.0, ga=20.0)
    ops = CudaOps()
    B, T = 256, 6
    lo = torch.randn((B, T), device=dev, requires_grad=True)
    sh = torch.tanh(torch.randn((B, T, 2), device=dev)).requires_grad_(True)
    sc = torch.sigmoid(torch.randn((B, T, 1), device=dev) - 1).requires_grad_(True)

    def asr():
        per_image, margin, _ = ops.asr(cfg, lo, sh, sc)
        (per_image.mean() + margin).backward()
    out["asr_reg_fwd_bwd_us_B256_T6_eager"] = timeit(asr, 100)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        asr()
    out["asr_reg_fwd_bwd_us_B256_T6_graph"] = timeit(g.replay, 200)
    # same at a 16k batch with the count penalties on (3 launches: column sums, forward, backward)
    cfg2 = config_from_flags("mnist", "13", gm=100.0, gne=10.0)
    lo2 = torch.randn((16384, T), device=dev, requires_grad=True)
    sh2 = torch.tanh(torch.randn((16384, T, 2), device=dev)).requires_grad_(True)
    sc2 = torch.sigmoid(torch.randn((16384, T, 1), device=dev) - 1).requires_grad_(True)

    def asr2():
        per_image, margin, _ = ops.asr(cfg2, lo2, sh2, sc2)
        (per_image.mean() + margin).backward()
    out["asr_reg_fwd_bwd_us_B16384_T6_eager"] = timeit(asr2, 50)
    # reconstruction loss at the headline canvas size
    Bc, P = 16384, 256 * 256
    canvas = (torch.rand((Bc, P), device=dev) * 1.2).requires_grad_(True)
    images = torch.rand((Bc, P), device=dev)
    gl = torch.rand(Bc, device=dev)
    loss = M.reconstruction_loss(canvas, images)[0]
    t_f = timeit(lambda: M.reconstruction_loss(canvas, images), 10)
    t_b = timeit(lambda: torch.autograd.grad(loss, canvas, gl, retain_graph=True), 10)
    out["bce_fwd"] = dict(us=t_f, gbs=8.0 * Bc * P / (t_f * 1e-6) / 1e9, frac=8.0 * Bc * P / (t_f * 1e-6) / 1e9 / peak,
                          bytes_per_pixel=8, shape=[Bc, P])
    out["bce_bwd"] = dict(us=t_b, gbs=12.0 * Bc * P / (t_b * 1e-6) / 1e9, frac=12.0 * Bc * P / (t_b * 1e-6) / 1e9 / peak,
                          bytes_per_pixel=12, shape=[Bc, P])
    out["general_affine"] = general_affine_section(dev, timeit)
    out["detection"] = detection_section(dev, timeit)
    out["dataset"] = dataset_section(dev, timeit)
    return out


def general_affine_section(dev, timeit):
    """The cold path: rotated thetas (t01, t10 != 0) and three channels take the per-pixel forward and the scatter-form
    backward (warp-aggregated red.global.add, csrc/mog_stn_warp.cuh: bwd_general_image).  Read direction 256x256 -> 64x64,
    4096 canvases; the separable kernels on the same shapes are timed beside it."""
    import torch
    from mog_asr_b200 import _lib, synth
    L = _lib.load()
    peak, _ = peak_hbm()
    B, cs, gs = 4096, 256, 64
    s_, x_, y_ = synth.sxy_prior_like(B, seed=77)
    phi = np.random.default_rng(78).uniform(-np.pi / 6, np.pi / 6, B).astype(np.float32)
    rot = np.stack([s_ * np.cos(phi), -s_ * np.sin(phi), x_, s_ * np.sin(phi), s_ * np.cos(phi), y_], 1).astype(np.float32)
    sep = synth.theta_read(s_, x_, y_)
    out = {}
    st = torch.cuda.current_stream(dev).cuda_stream
    for C in (1, 3):
        U = torch.rand((B, cs, cs, C), device=dev)
        g = torch.randn((B, gs, gs, C), device=dev)
        o, dU, dth = torch.empty((B, gs, gs, C), device=dev), torch.empty_like(U), torch.empty((B, 6), device=dev)
        for name, th in (("rotated", rot), ("axis_aligned", sep)):
            if name == "axis_aligned" and C != 1:
                continue                                   # (C > 1 always takes the general path)
            t = torch.tensor(th, device=dev)
            f = lambda: _lib.check(L.mog_stn_forward(U.data_ptr(), t.data_ptr(), o.data_ptr(), B, cs, cs, C, gs, gs, 1, st), "fwd")
            b = lambda: _lib.check(L.mog_stn_backward(U.data_ptr(), t.data_ptr(), g.data_ptr(), dU.data_ptr(), dth.data_ptr(), B, cs, cs, C,
                                                      gs, gs, 1, st), "bwd")
            tf_, tb_ = timeit(f, 5), timeit(b, 5)
            out[f"{name}_C{C}"] = dict(fwd_us=tf_, bwd_us=tb_, glimpses_per_s_fwd_bwd=B / ((tf_ + tb_) * 1e-6),
                                       bwd_write_gbs=4.0 * B * cs * cs * C / (tb_ * 1e-6) / 1e9,
                                       bwd_frac_of_peak_by_dU_bytes=4.0 * B * cs * cs * C / (tb_ * 1e-6) / 1e9 / peak)
        del U, g, o, dU
        torch.cuda.empty_cache()
    # magnifying direction (a 64 x 64 window written onto a 256 x 256 canvas, full-cover scale: ~3.6 output pixels per source
    # pixel): the case warp aggregation is for -- every source pixel receives many lanes' contributions
    s2, x2, y2 = synth.sxy_full_cover(B, seed=79)
    inv = 1.0 / s2
    rotw = np.stack([inv * np.cos(phi), inv * np.sin(phi), -(x2 * np.cos(phi) + y2 * np.sin(phi)) * inv,
                     -inv * np.sin(phi), inv * np.cos(phi), (x2 * np.sin(phi) - y2 * np.cos(phi)) * inv], 1).astype(np.float32)
    W = torch.rand((B, gs, gs, 1), device=dev)
    gw = torch.randn((B, cs, cs, 1), device=dev)
    ow, dW, dth = torch.empty((B, cs, cs, 1), device=dev), torch.empty_like(W), torch.empty((B, 6), device=dev)
    t = torch.tensor(rotw, device=dev)
    f = lambda: _lib.check(L.mog_stn_forward(W.data_ptr(), t.data_ptr(), ow.data_ptr(), B, gs, gs, 1, cs, cs, 1, st), "fwd")
    b = lambda: _lib.check(L.mog_stn_backward(W.data_ptr(), t.data_ptr(), gw.data_ptr(), dW.data_ptr(), dth.data_ptr(), B, gs, gs, 1,
                                              cs, cs, 1, st), "bwd")
    tf_, tb_ = timeit(f, 3), timeit(b, 3)
    out["rotated_write_full_cover_C1"] = dict(fwd_us=tf_, bwd_us=tb_, glimpses_per_s_fwd_bwd=B / ((tf_ + tb_) * 1e-6),
                                              bwd_read_gbs=4.0 * B * cs * cs / (tb_ * 1e-6) / 1e9)
    out["workload"] = (f"read {cs}x{cs} -> {gs}x{gs} and (write, full-cover scale) {gs}x{gs} -> {cs}x{cs}, {B} canvases, "
                       "rotation uniform in +-30 degrees")
    return out


def dataset_section(dev, timeit):
    """On-device synthetic feeder (multi_mnist.py:110-221 placement + paste through the sampler): canvases per second
    for 50x50 Multi-MNIST-like batches of 4096, next to this repo's numpy generator on one host core."""
    import torch
    from mog_asr_b200 import synth
    from mog_asr_b200.dataset import DeviceMultiObjectDataset, default_sprites
    ds = DeviceMultiObjectDataset(default_sprites(256, 28, seed=0), 50, (1, 2, 3), (17, 23), mode="disjoint", seed=5, device=dev)
    B = 4096
    k = [0]

    def gen():
        k[0] += 1
        return ds.batch(k[0], B)
    t_us = timeit(gen, 20)
    t_place = timeit(lambda: ds.place(0, B), 50)
    t0 = time.perf_counter()
    synth.multi_object_canvases(256, 50, 28, (1, 2, 3), seed=0)
    t_host = (time.perf_counter() - t0) / 256
    return dict(batch=B, us_per_batch=t_us, canvases_per_s=B / (t_us * 1e-6), placement_kernel_us=t_place,
                host_numpy_generator_canvases_per_s=1.0 / t_host, host_cores=1)


def detection_section(dev, timeit):
    """Detection metrics (evaluation_detection.py:29-98) for a 10 000-image evaluation set, 3 ground-truth and up to 3
    inferred boxes: the kernel alone, the reference-signature call (ragged host lists in, means out) and the CPU port
    of the reference loop on a 2 000-image sample (cpu_baseline leg: the only place the oracle is timed)."""
    import numpy as np
    import torch
    from mog_asr_b200 import detection
    rng = np.random.default_rng(0)
    n, cs, G, T = 10000, 50, 3, 3
    gt_num, inf_num = rng.integers(0, G + 1, n), rng.integers(0, T + 1, n)
    wh = rng.integers(8, 24, (n, G, 2))
    xy = (rng.random((n, G, 2)) * (cs - wh)).astype(np.int64)
    pos = [xy[k, :gt_num[k]].reshape(-1).tolist() for k in range(n)]
    size = [wh[k, :gt_num[k]].reshape(-1).tolist() for k in range(n)]
    shifts = np.tanh(rng.normal(0, 0.5, (n, T, 2))).astype(np.float32)
    scales = (1 / (1 + np.exp(-rng.normal(-1, 0.5, (n, T, 1))))).astype(np.float32)
    d = lambda a: torch.as_tensor(a).to(dev)
    P, S, num = detection.pack_ground_truth(pos, size)
    dP, dS, dnum, dsh, dsc, dinf = d(P), d(S), d(num), d(shifts).double(), d(scales).double(), d(inf_num.astype(np.int32))
    t_kernel = timeit(lambda: detection.detection_metrics(dP, dS, dnum, dsh, dsc, dinf, cs), 50)
    t0 = time.perf_counter()
    got = detection.evaluation(pos, size, shifts, scales, inf_num, csize=cs, device=dev)
    t_call = time.perf_counter() - t0
    from oracle import detection_ref                       # CPU baseline leg
    m = 2000
    t0 = time.perf_counter()
    want = detection_ref.evaluation(pos[:m], size[:m], shifts[:m], scales[:m], inf_num[:m], csize=cs)
    t_cpu = time.perf_counter() - t0
    chk = detection.evaluation(pos[:m], size[:m], shifts[:m], scales[:m], inf_num[:m], csize=cs, device=dev)
    same = all(np.array_equal(np.asarray(a), np.asarray(b)) for a, b in zip(chk[:4], want[:4])) and abs(chk[4] - want[4]) < 1e-14
    return dict(images=n, kernel_us=t_kernel, images_per_s_kernel=n / (t_kernel * 1e-6), call_ms_host_lists=t_call * 1e3,
                images_per_s_call=n / t_call, precision_at_0p5=float(got[0][0]),
                cpu_baseline=dict(value=m / t_cpu, unit="images/s", cores=1, kind="port", sample=f"{m} images, oracle/detection_ref.py"),
                matches_cpu_port=bool(same))


def train_section(a, dev, world, pg, rank):
    """Secondary metric of BASELINE.json: AIR-ASR training images/sec (configs 2-4) around the same kernels."""
    from mog_asr_b200.air import bench_train
    out = {}
    r = bench_train.run("C4", dev, steps=10, warmup=3, process_group=pg, always_max_steps=True, graph=True)
    out["C4_global4096"] = r
    if world > 1:
        try:   # multi-GPU correctness on this very hardware: all-reduced gradient vs the single-process global-batch gradient
            out["dp_check"] = bench_train.dp_check(dev, pg)
        except Exception as e:
            out["dp_check"] = dict(error=f"{type(e).__name__}: {e}")
        # the same model with the per-GPU work held at 4096 images (weak scaling): separates the all-reduce cost from
        # the fixed per-step launch chain that bounds the strong-scaling line above
        out["C4_weak_4096_per_gpu"] = bench_train.run("C4", dev, steps=10, warmup=3, process_group=pg, always_max_steps=True,
                                                      graph=True, per_rank_batch=4096)
    if world == 1:
        for name in ("C2", "C3"):
            out[name + "_graph"] = bench_train.run(name, dev, steps=10, warmup=3, always_max_steps=True, graph=True)
            out[name + "_eager_reference_loop"] = bench_train.run(name, dev, steps=10, warmup=3)
        if not a.no_cpu:
            out["cpu_port_C2"] = train_cpu_baseline()
    return out


def train_cpu_baseline():
    """C2 step (batch 64) with the oracle's operators on the host cores (torch-CPU, all threads)."""
    import torch
    from mog_asr_b200.air import Trainer, bench_train, config_from_flags
    from oracle.air_ops import OracleOps
    flags, gb = bench_train.CONFIGS["C2"]
    cfg = config_from_flags(**flags)
    torch.set_num_threads(host_threads())
    tr = Trainer(cfg, "cpu", ops=OracleOps())
    images = bench_train.synthetic_batch(cfg, gb, 0, "cpu")
    tr.step(images)
    t0 = time.perf_counter()
    n = 3
    for _ in range(n):
        tr.step(images)
    dt = (time.perf_counter() - t0) / n
    return dict(images_per_sec=gb / dt, ms_per_step=dt * 1e3, global_batch=gb, cores=torch.get_num_threads(), kind="port",
                sample=f"{n} steps of config C2 (batch {gb}) with oracle/air_ops.py on torch-CPU")


def trace(msg):
    """progress marker on stderr (the JSON line is the only thing that goes to stdout)"""
    print(f"[bench rank {os.environ.get('RANK', '0')} +{time.perf_counter() - _T0:.1f}s] {msg}", file=sys.stderr, flush=True)


_T0 = time.perf_counter()


def run_ours(a):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: this path has no CPU fallback (use --impl reference for the CPU arm)")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    import mog_asr_b200 as M  # noqa: F401
    from mog_asr_b200 import _lib
    _lib.load()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    trace("building workload")
    wl = GpuWorkload(a, dev, seed=10 + rank)
    trace("warm-up")
    sampler = ClockSampler(local)
    sampler.start()
    for _ in range(max(a.warmup, 3)):
        wl.step()
    barrier()
    events = {k: [] for k in wl.kinds}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    tc0 = time.perf_counter()
    e0.record()
    for _ in range(a.steps):
        wl.step(events)
    e1.record()
    barrier()
    tc1 = time.perf_counter()
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    trace(f"timed region done: {ms_total / a.steps:.3f} ms/step")
    if a.dump_outputs and rank == 0:
        dump_outputs(wl, a.dump_outputs)
    ms_per_step = ms_total / a.steps
    glimpses_per_step = a.batch * 2 * AIR_STEPS * world
    value = glimpses_per_step / (ms_per_step * 1e-3)

    kern_ms = {k: float(np.mean([x.elapsed_time(y) for x, y in events[k]])) for k in wl.kinds}
    kern_share = {k: kern_ms[k] * AIR_STEPS / ms_per_step for k in wl.kinds}

    # e2e: host buffers through the C ABI
    e2e = None
    e2e_launches = 0
    if not a.no_e2e:
        e_steps = 2 if a.batch * a.canvas ** 2 > (1 << 28) else max(2, a.steps // 10)
        trace("e2e leg")
        dt, h2d, d2h, e2e_launches, api = e2e_measure(a, dev, max(e_steps, 3), 1)
        trace("e2e done")
        barrier()
        dt = max_over_ranks(dt)
        e2e = dict(value=a.e2e_batch * 2 * AIR_STEPS * world / dt, unit=UNIT, h2d_bytes_per_step=int(h2d),
                   d2h_bytes_per_step=int(d2h), ms_per_step=dt * 1e3, steps=max(e_steps, 3), batch_per_gpu=a.e2e_batch, api=api)
        # the same glimpses with every write step's 256x256 canvas and gradient crossing the bus separately (round-1/2 form)
        dt2, h2d2, d2h2, _, api2 = e2e_measure(a, dev, 1, 1, composite=False)
        barrier()
        dt2 = max_over_ranks(dt2)
        e2e["separate_write_canvases"] = dict(value=a.e2e_batch * 2 * AIR_STEPS * world / dt2, unit=UNIT, h2d_bytes_per_step=int(h2d2),
                                              d2h_bytes_per_step=int(d2h2), ms_per_step=dt2 * 1e3, steps=1, api=api2)
    tc2 = time.perf_counter()
    sampler.stop_flag = True
    clocks = sampler.summary(tc0, tc2 if e2e else tc1)

    if rank == 0:
        peak, peak_src = peak_hbm()
        abytes = wl.algorithmic_bytes()
        dom = max(wl.kinds, key=lambda k: kern_ms[k])
        kernels = {k: dict(ms=kern_ms[k], share_of_step=kern_share[k], alg_bytes_per_launch=abytes[k],
                           achieved_gbs=abytes[k] / (kern_ms[k] * 1e-3) / 1e9,
                           frac=abytes[k] / (kern_ms[k] * 1e-3) / 1e9 / peak) for k in wl.kinds}
        nxc = lambda w: 1 if w <= 32 else (2 if w <= 64 else 4)
        sym = dict(read_fwd="stn_fwd_warp_kernel<false>", write_fwd="stn_fwd_warp_kernel<false>",
                   read_bwd=f"stn_bwd_warp_kernel<false,{nxc(a.canvas)}>",
                   write_bwd=("stn_bwd_cta_kernel<false,8,%d>" % (1 if a.glimpse ** 2 > 1024 else 2)) if (a.canvas >= 192 and a.glimpse <= 64)
                   else f"stn_bwd_warp_kernel<false,{nxc(a.glimpse)}>")
        # physical DRAM bytes per launch of ALL four kernels, from the ncu capture committed with this bench line
        # (tools/traffic_capture.py: dram__bytes_read.sum + dram__bytes_write.sum, same cell, same batch)
        traffic, traffic_src, tj = None, None, None
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "traffic_latest.json")))
            if tj["cell"] != dict(canvas=a.canvas, glimpse=a.glimpse, regime=a.regime, batch=a.batch):
                tj = None
        except Exception:
            tj = None
        if tj is not None:
            traffic, traffic_src = tj["bytes_per_launch"][dom], tj["source"]
            for k in wl.kinds:
                kernels[k]["traffic_bytes_per_launch"] = tj["bytes_per_launch"][k]
                kernels[k]["frac_physical"] = tj["bytes_per_launch"][k] / (kern_ms[k] * 1e-3) / 1e9 / peak
        # the AIR read call site asks for dtheta only (air_number_bbox_location.py:534-542): reported beside the dU + dtheta form
        evs = []
        for t in range(AIR_STEPS):
            e0_, e1_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0_.record(); wl.launch("read_bwd_dtheta", t); e1_.record()
            evs.append((e0_, e1_))
        torch.cuda.synchronize(dev)
        ms_dt = float(np.mean([x.elapsed_time(y) for x, y in evs]))
        kernels["read_bwd_dtheta_only"] = dict(ms=ms_dt, alg_bytes_per_launch=abytes["read_bwd_dtheta"],
                                               achieved_gbs=abytes["read_bwd_dtheta"] / (ms_dt * 1e-3) / 1e9,
                                               frac=abytes["read_bwd_dtheta"] / (ms_dt * 1e-3) / 1e9 / peak,
                                               note="not part of the timed step: the AIR-faithful read backward (no dU)")
        roofline = dict(bound="hbm", kernel=f"{sym[dom]} ({dom})", achieved=kernels[dom]["achieved_gbs"], peak=peak,
                        unit="GB/s", frac=kernels[dom]["frac"], traffic=traffic, traffic_source=traffic_src,
                        algorithmic_bytes_per_launch=abytes[dom], peak_source=peak_src,
                        note="algorithmic bytes: fwd 4(F+O)+24, bwd 4(G+F+S)+48 with G = the in-range part of the upstream gradient "
                             "(SURVEY 8(d) charges all of O; survey_bytes_per_launch keeps that figure); frac_physical uses measured DRAM bytes",
                        survey_bytes_per_launch=getattr(wl, "survey_bytes", None),
                        step_alg_gbs=sum(abytes[k] for k in wl.kinds) * AIR_STEPS / (ms_per_step * 1e-3) / 1e9,
                        kernels=kernels)
        roofline["step_frac"] = roofline["step_alg_gbs"] / peak
        if tj is not None:
            roofline["step_physical_gbs"] = sum(tj["bytes_per_launch"][k] for k in wl.kinds) * AIR_STEPS / (ms_per_step * 1e-3) / 1e9
            roofline["step_frac_physical"] = roofline["step_physical_gbs"] / peak
        line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=a.steps, warmup=max(a.warmup, 3),
                    ms_per_step=ms_per_step, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32",
                    data="synthetic",
                    config=config_dict(a),
                    roofline=roofline, clocks=clocks, gpu_launches=4 * AIR_STEPS * a.steps)
        if e2e:
            line["e2e"] = e2e
            line["e2e_gpu_launches"] = e2e_launches * e2e["steps"]
        if world == 1 and not a.no_cpu:
            cb, _ = cpu_measure(a, 3, 1, a.cpu_sample)
            line["cpu_baseline"] = cb
        if world == 1:
            try:
                line["config1"] = config1_section(dev, a.no_cpu)
            except Exception as e:
                line["config1"] = dict(error=f"{type(e).__name__}: {e}")
            try:
                del wl
                torch.cuda.empty_cache()
                line["aux_kernels"] = aux_section(dev)
            except Exception as e:
                line["aux_kernels"] = dict(error=f"{type(e).__name__}: {e}")
    train = None
    if not a.no_train:
        trace("train section")
        try:
            train = train_section(a, dev, world, dist.group.WORLD if world > 1 else None, rank)
        except Exception as e:  # never lose the headline line to the secondary metric
            train = dict(error=f"{type(e).__name__}: {e}")
    trace("printing")
    if rank == 0:
        if train is not None:
            line["train"] = train
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_sweep(a):
    """Every cell of BASELINE config 5 on one GPU: canvas {50,64,128,256} x glimpse {28,64} (glimpse < canvas),
    theta regimes prior-like / full-cover, read and write directions; writes profiles/sweep_<tag>.json."""
    import copy
    import torch
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    peak, peak_src = peak_hbm()
    rows = []
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", f"traffic_{a.tag or 'latest'}_sweep.json")))
    except Exception:
        traffic = {}
    for canvas in (50, 64, 128, 256):
        for glimpse in (28, 64):
            if glimpse >= canvas:
                continue
            for regime in ("prior", "full"):
                c = copy.copy(a)
                c.canvas, c.glimpse, c.regime = canvas, glimpse, regime
                wl = GpuWorkload(c, dev, seed=10)
                for _ in range(3):
                    wl.step()
                torch.cuda.synchronize(dev)
                events = {k: [] for k in wl.kinds}
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(a.steps):
                    wl.step(events)
                e1.record()
                torch.cuda.synchronize(dev)
                ms = e0.elapsed_time(e1) / a.steps
                kern_ms = {k: float(np.mean([x.elapsed_time(y) for x, y in events[k]])) for k in wl.kinds}
                ab = wl.algorithmic_bytes()
                row = dict(canvas=canvas, glimpse=glimpse, regime=regime, batch=c.batch, ms_per_step=ms,
                           glimpses_per_sec=c.batch * 2 * AIR_STEPS / (ms * 1e-3),
                           step_alg_gbs=sum(ab[k] for k in wl.kinds) * AIR_STEPS / (ms * 1e-3) / 1e9,
                           kernels={k: dict(us=kern_ms[k] * 1e3, alg_mb=ab[k] / 1e6, gbs=ab[k] / (kern_ms[k] * 1e-3) / 1e9,
                                            frac=ab[k] / (kern_ms[k] * 1e-3) / 1e9 / peak) for k in wl.kinds})
                row["step_frac"] = row["step_alg_gbs"] / peak
                tcell = traffic.get(f"{canvas}:{glimpse}:{regime}")
                if tcell and tcell["cell"]["batch"] == c.batch:     # measured DRAM bytes per launch (tools/traffic_capture.py under ncu)
                    for k in wl.kinds:
                        row["kernels"][k]["traffic_mb"] = tcell["bytes_per_launch"][k] / 1e6
                        row["kernels"][k]["frac_physical"] = tcell["bytes_per_launch"][k] / (kern_ms[k] * 1e-3) / 1e9 / peak
                    row["step_physical_gbs"] = sum(tcell["bytes_per_launch"][k] for k in wl.kinds) * AIR_STEPS / (ms * 1e-3) / 1e9
                    row["step_frac_physical"] = row["step_physical_gbs"] / peak
                rows.append(row)
                emit(row)
                del wl
                torch.cuda.empty_cache()
    out = os.path.join(ROOT, "profiles", f"sweep_{a.tag or 'latest'}.json")
    with open(out, "w") as f:
        json.dump(dict(peak_gbs=peak, peak_source=peak_src, steps=a.steps, cells=rows), f, indent=1)


_REAL_STDOUT = None


def protect_stdout():
    """The contract is ONE JSON line on stdout.  Libraries print there too (NCCL: "NCCL version ..."), so fd 1 is
    pointed at stderr for the whole run and the JSON line goes to the saved descriptor."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def emit(line: dict):
    _REAL_STDOUT.write(json.dumps(line) + "\n")
    _REAL_STDOUT.flush()


def main():
    a = parse_args()
    protect_stdout()
    if a.cpu_sample <= 0:   # ~7e-8 s per output pixel and core for fwd+bwd of the C port -> about a second per step
        px = AIR_STEPS * (a.glimpse ** 2 + 2 * a.canvas ** 2)
        a.cpu_sample = int(max(64, min(1024, 2 ** round(np.log2(16 * 1.0 / (7e-8 * px))))))
    if a.e2e_batch <= 0:
        # the full batch on one GPU; with N ranks on one host the pinned arrays (4 canvases' worth per image and rank)
        # would not fit, so every rank takes batch/N images: the leg is host/PCIe-bound and its rate per byte is the same
        world = int(os.environ.get("WORLD_SIZE", "1"))
        a.e2e_batch = a.batch if world == 1 else max(2048, a.batch // world)
    if a.impl == "reference":
        run_reference(a)
    elif a.sweep:
        run_sweep(a)
    else:
        run_ours(a)


if __name__ == "__main__":
    main()
