"""GPU parity of the kernels that run around the sampler in every AIR training step -- the fused (mean, log-variance) heads
(csrc/mog_air_head.cu), the dense-layer epilogues, per-step elementwise kernels and KL terms (csrc/mog_air.cu) and the
reconstruction loss (csrc/mog_bce.cu) -- against fp64 restatements of the formulas in include/mogstn.h, evaluated on the CPU.

Every launcher caps its grid at a multiple of the SM count.  Past one grid pass a warp or thread handles several rows and
carries its per-lane partials from one row to the next, so the sizes below are derived from the device's SM count with the
launchers' multipliers, and every case meant to take several passes asserts that it does.  The head runs in each of its
four instantiations (hidden 16, 32, 64, 128).  Every output the header says is fully overwritten is pre-filled with NaN,
so an element a kernel never writes fails the comparison.  The C ABI is called directly, on the current stream.

Tolerances: the head's mean, log-variance and gradients are held to ``GRAD_RTOL`` relative to the sum of |terms| entering
each entry (DESIGN.md section 4); values computed from the kernel's own fp32 intermediates to a few ulp; the per-step
kernels and the reconstruction loss to the bounds of tests/test_air_fused_gpu.py and tests/test_bce_gpu.py, taken
relative to the sum of |terms| where, among this many draws, the terms of an entry cancel.  Derivatives of tanh and
sigmoid are taken from the saved output, as the kernels and TF's TanhGrad / SigmoidGrad do."""
import numpy as np
import pytest
import torch
from scipy import special

from mog_asr_b200 import _lib
from oracle import bce_ref
from tests import helpers as H

pytestmark = pytest.mark.gpu

EPS32 = H.EPS32
FLT_MIN = 2.0 ** -126   # absolute floor of the ulp bounds: below it an fp32 result may be denormal or flushed to zero


# elements one grid pass covers, with the multipliers of the launchers
def head_pass(dev):      # launch_head: 4 CTAs per SM x 8 warps, one row per warp
    return torch.cuda.get_device_properties(dev).multi_processor_count * 4 * 8


def elem_pass(dev):      # air_blocks: 8 CTAs per SM x 256 threads, one element per thread
    return torch.cuda.get_device_properties(dev).multi_processor_count * 8 * 256


def bce_fwd_pass(dev):   # mog_bce_recon_forward: 8 CTAs per SM x 8 warps, one image per warp
    return torch.cuda.get_device_properties(dev).multi_processor_count * 8 * 8


def bce_bwd_pass(dev):   # mog_bce_recon_backward: 8 CTAs per SM, one image per CTA
    return torch.cuda.get_device_properties(dev).multi_processor_count * 8


def ptr(t):
    return t.data_ptr() if t is not None else None


def call(fn, *args):
    rc = fn(*args, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert rc == 0, _lib.last_error()


def nan_buffer(shape, dev):
    return torch.full(shape, float("nan"), device=dev)


def to_dev(t, dev):
    return t.to(dev) if t is not None else None


def f64(t):
    return t.detach().cpu().double()


def ulp_excess(got, ref, scale, ulps):
    """max of |got - ref| / (ulps * 2^-23 * scale + FLT_MIN); <= 1 passes, a NaN in got fails"""
    err = (f64(got) - ref).abs() / (ulps * EPS32 * scale + FLT_MIN)
    return float(torch.nan_to_num(err, nan=float("inf")).max())


def close_excess(got, ref, rtol, atol):
    """max of |got - ref| / (atol + rtol * |ref|): the bound of assert_allclose; <= 1 passes, a NaN in got fails"""
    err = (f64(got) - ref).abs() / (atol + rtol * ref.abs())
    return float(torch.nan_to_num(err, nan=float("inf")).max())


def grad_excess(got, ref, absterms):
    return H.grad_excess(f64(got).numpy(), ref.numpy(), absterms.numpy())


# ---------------------------------------------------------------------------------------------------------------------
# (mean, log-variance) heads: mog_air_head_forward / _backward
# ---------------------------------------------------------------------------------------------------------------------
# (hidden, S skip inputs, O outputs, act, K): launch_head instantiates air_head_kernel<NQ> with NQ = 2 * hidden / 32; every S,
# O and act appears in at least two classes.  An odd K puts the skip columns of w1 at an odd offset of the row.
HEAD_CLASSES = [
    pytest.param(16, 1, 2, 0, 37, id="h16-s1-o2-none-K37"),
    pytest.param(16, 2, 1, 2, 256, id="h16-s2-o1-sigmoid"),
    pytest.param(32, 0, 1, 1, 256, id="h32-s0-o1-tanh"),
    pytest.param(32, 2, 2, 0, 37, id="h32-s2-o2-none-K37"),
    pytest.param(64, 0, 2, 1, 256, id="h64-shift-head"),     # the model's shift head (:424-436)
    pytest.param(64, 2, 1, 2, 256, id="h64-scale-head"),     # the model's scale head, fed the shift sample (:439-459)
    pytest.param(128, 1, 1, 0, 37, id="h128-s1-o1-none-K37"),
    pytest.param(128, 2, 2, 1, 37, id="h128-s2-o2-tanh-K37"),
]
# B = 1 and 5: one CTA with idle warps whose zero partials enter the reduction; one pass exactly: one row per warp;
# multi_pass: about three passes and a ragged remainder, so every warp carries its partials over several rows
HEAD_ROWS = ["B1", "B5", "one_pass", "multi_pass"]
G_NAMES = ("g_mean", "g_logvar", "g_latent", "g_squashed")
HEAD_P = 0.375   # what the accumulated parameter-gradient buffers hold before a backward call


def dyadic(shape, gen, lim):
    """multiples of 2^-10 in [-lim, lim]"""
    m = int(lim * 1024)
    return torch.randint(-m, m + 1, shape, generator=gen).float() / 1024


def head_inputs(B, h, K, S, O, seed):
    """Dyadic inputs: the first-layer pre-activation v = pre1 + b1 + sum_s skip_s * w1s_s is a multiple of 2^-20 below 16,
    exact in fp32, so the relu mask is the same in fp32 and fp64.  About 5 % of the entries of pre1 are planted to make v
    exactly 0.  The columns of w1 before K are NaN: only the skip columns may be read."""
    gen = torch.Generator().manual_seed(seed)
    a = {"pre1": dyadic((B, 2 * h), gen, 2), "skip": dyadic((B, S), gen, 2) if S else None, "eps": dyadic((B, O), gen, 2)}
    for br in "mv":
        w1 = torch.full((h, K + S), float("nan"))
        w1[:, K:] = dyadic((h, S), gen, 2)
        a["w1" + br] = w1
        a["b1" + br] = dyadic((h,), gen, 2)
        a["w2" + br] = dyadic((O, h + S), gen, h ** -0.5)   # keeps logvar within a few units
        a["b2" + br] = dyadic((O,), gen, 0.5)
    rest = torch.cat([a["b1m"], a["b1v"]]).double().expand(B, 2 * h).clone()
    if S:
        rest += a["skip"].double() @ torch.cat([a["w1m"][:, K:], a["w1v"][:, K:]]).double().T
    zero = torch.rand((B, 2 * h), generator=gen) < 0.05
    a["pre1"][zero] = (-rest[zero]).float()
    for k in G_NAMES:
        a[k] = dyadic((B, O), gen, 2)
    return a, zero


def head_forward_ref(a, h, K, S):
    """mean, logvar and the sum of |terms| of each, plus the first layer's pre-activations v* and outputs h*, in fp64"""
    d = {k: v.double() for k, v in a.items() if v is not None}
    B = d["pre1"].shape[0]
    sk = d["skip"] if S else torch.zeros(B, 0, dtype=torch.float64)
    f = {"skip": sk}
    for br, cols, name in (("m", slice(0, h), "mean"), ("v", slice(h, 2 * h), "logvar")):
        v = d["pre1"][:, cols] + d["b1" + br] + sk @ d["w1" + br][:, K:].T
        hid = v.clamp_min(0.0)
        w2, b2 = d["w2" + br], d["b2" + br]
        f["v" + br], f["h" + br] = v, hid
        f[name] = hid @ w2[:, :h].T + sk @ w2[:, h:].T + b2
        f["A" + name] = hid @ w2[:, :h].abs().T + sk.abs() @ w2[:, h:].abs().T + b2.abs()
    return f


def head_backward_ref(a, f, logvar, squashed, grads, h, K, act):
    """The fp64 chain rule, and the sum of |terms| entering each entry, for the gradient inputs named in ``grads``.
    tanh' and sigmoid' are taken from the saved squashed output, as TF's TanhGrad / SigmoidGrad do."""
    d = {k: v.double() for k, v in a.items() if v is not None}
    eps, sk = d["eps"], f["skip"]
    zero = torch.zeros_like(eps)
    g = {k: d[k] if k in grads else zero for k in G_NAMES}
    if act == 1:
        sq = f64(squashed)
        dsq, adsq = 1 - sq * sq, 1 + sq * sq
    elif act == 2:
        sq = f64(squashed)
        dsq, adsq = sq * (1 - sq), sq.abs() * (1 + sq.abs())
    else:
        dsq = adsq = zero
    dl = g["g_latent"] + g["g_squashed"] * dsq
    adl = g["g_latent"].abs() + g["g_squashed"].abs() * adsq
    half_sigma = 0.5 * torch.exp(0.5 * f64(logvar))
    dy = {"m": g["g_mean"] + dl, "v": g["g_logvar"] + dl * eps * half_sigma}
    ady = {"m": g["g_mean"].abs() + adl, "v": g["g_logvar"].abs() + adl * eps.abs() * half_sigma}
    r, dp, adp = {}, {}, {}
    for br in "mv":
        w2 = d["w2" + br]
        mask = (f["v" + br] > 0).double()                     # relu'(0) = 0
        dp[br] = (dy[br] @ w2[:, :h]) * mask
        adp[br] = (ady[br] @ w2[:, :h].abs()) * mask
        r["gw2" + br] = torch.cat([dy[br].T @ f["h" + br], dy[br].T @ sk], 1)
        r["Agw2" + br] = torch.cat([ady[br].T @ f["h" + br], ady[br].T @ sk.abs()], 1)
        r["gb2" + br], r["Agb2" + br] = dy[br].sum(0), ady[br].sum(0)
    r["dpre1"], r["Adpre1"] = torch.cat([dp["m"], dp["v"]], 1), torch.cat([adp["m"], adp["v"]], 1)
    r["dskip"] = sum(dp[br] @ d["w1" + br][:, K:] + dy[br] @ d["w2" + br][:, h:] for br in "mv")
    r["Adskip"] = sum(adp[br] @ d["w1" + br][:, K:].abs() + ady[br] @ d["w2" + br][:, h:].abs() for br in "mv")
    return r


@pytest.mark.parametrize("rows", HEAD_ROWS)
@pytest.mark.parametrize("hidden,S,O,act,K", HEAD_CLASSES)
def test_head_matches_fp64(cuda_device, hidden, S, O, act, K, rows):
    """mog_air_head_forward / _backward against the fp64 formulas of the header: mean and logvar, dpre1, dskip and the
    accumulated second-layer parameter gradients within GRAD_RTOL of the sum of |terms|; latent and squashed within 4 ulp of
    the formula applied to the kernel's own mean and logvar; dpre1 exactly 0 where v = 0; each gradient input alone and all
    together; g_squashed ignored when act = 0; dpre1 and dskip the same bits on every run and without dskip; the parameter
    gradients added to what their buffers hold, twice over for two calls."""
    L = _lib.load()
    dev = cuda_device
    h = hidden
    per_pass = head_pass(dev)
    B = {"B1": 1, "B5": 5, "one_pass": per_pass, "multi_pass": 3 * per_pass + 1237}[rows]
    if rows == "multi_pass":
        assert B > 3 * per_pass and B % 8 != 0
    a, zero = head_inputs(B, h, K, S, O, seed=h * 100 + S * 10 + O + B)
    t = {k: to_dev(v, dev) for k, v in a.items()}

    mean, logvar, latent = (nan_buffer((B, O), dev) for _ in range(3))
    squashed = nan_buffer((B, O), dev) if act else None
    call(L.mog_air_head_forward, *(ptr(t[k]) for k in ("pre1", "skip", "eps", "w1m", "b1m", "w1v", "b1v", "w2m", "b2m", "w2v", "b2v")),
         B, h, K, S, O, act, ptr(mean), ptr(logvar), ptr(latent), ptr(squashed))
    f = head_forward_ref(a, h, K, S)
    assert grad_excess(mean, f["mean"], f["Amean"]) <= 1.0
    assert grad_excess(logvar, f["logvar"], f["Alogvar"]) <= 1.0
    m, lv, e = f64(mean), f64(logvar), a["eps"].double()
    noise = e * torch.exp(0.5 * lv)
    assert ulp_excess(latent, m + noise, m.abs() + noise.abs(), 4) <= 1.0
    if act:
        lat = f64(latent)
        ref = torch.tanh(lat) if act == 1 else torch.sigmoid(lat)
        assert ulp_excess(squashed, ref, ref.abs(), 4) <= 1.0

    def fresh_params():
        return {k: torch.full(shape, HEAD_P, device=dev)
                for k, shape in (("gw2m", (O, h + S)), ("gb2m", (O,)), ("gw2v", (O, h + S)), ("gb2v", (O,)))}

    def backward(grads, want_dskip=True, params=None):
        dpre1 = nan_buffer((B, 2 * h), dev)
        dskip = nan_buffer((B, S), dev) if S and want_dskip else None
        params = fresh_params() if params is None else params
        call(L.mog_air_head_backward, *(ptr(t[k]) for k in ("pre1", "skip", "eps", "w1m", "b1m", "w1v", "b1v", "w2m", "w2v")),
             ptr(logvar), ptr(squashed), *(ptr(t[k]) if k in grads else None for k in G_NAMES), B, h, K, S, O, act,
             ptr(dpre1), ptr(dskip), *(ptr(params[k]) for k in ("gw2m", "gb2m", "gw2v", "gb2v")))
        return dpre1, dskip, params

    def check(grads, dpre1, dskip, params, calls=1):
        r = head_backward_ref(a, f, logvar, squashed, grads, h, K, act)
        assert grad_excess(dpre1, r["dpre1"], r["Adpre1"]) <= 1.0, grads
        assert torch.all(dpre1.cpu()[zero] == 0), grads
        if S:
            assert grad_excess(dskip, r["dskip"], r["Adskip"]) <= 1.0, grads
        for k in ("gw2m", "gb2m", "gw2v", "gb2v"):
            assert grad_excess(params[k], HEAD_P + calls * r[k], HEAD_P + calls * r["A" + k]) <= 1.0, (grads, k)

    for grads in [(k,) for k in G_NAMES] + [G_NAMES]:
        dpre1, dskip, params = backward(grads)
        check(grads, dpre1, dskip, params)

    again = backward(G_NAMES)                                       # no atomics in dpre1 / dskip: the same bits
    assert torch.equal(again[0], dpre1)
    if S:
        assert torch.equal(again[1], dskip)
        assert torch.equal(backward(G_NAMES, want_dskip=False)[0], dpre1)
    if act == 0:
        plain = backward(G_NAMES[:3])
        assert torch.equal(plain[0], dpre1)
        if S:
            assert torch.equal(plain[1], dskip)

    params = backward(G_NAMES)[2]                                   # accumulated, not overwritten
    backward(G_NAMES, params=params)
    check(G_NAMES, dpre1, dskip, params, calls=2)


# ---------------------------------------------------------------------------------------------------------------------
# dense-layer epilogues: mog_air_bias_act_* and mog_air_bias_gauss_*
# ---------------------------------------------------------------------------------------------------------------------
ACTS = [pytest.param(0, id="none"), pytest.param(1, id="relu"), pytest.param(2, id="softplus"), pytest.param(3, id="sigmoid")]
# planted pre-activations: relu at 0 (both signs); softplus deep in the negative range, at and around its threshold 20
# (linear above); sigmoid where exp overflows or the result is denormal
EDGES = [0.0, -0.0, -30.0, -20.0, -10.0, -5.0, -2.0, 19.99, 20.0, float(np.nextafter(np.float32(20), np.float32(30))), 30.0,
         -90.0, 90.0]


def bias_act_inputs(B, N, seed):
    """pre [B][N] (bulk values spanning +-20) and bias [N]; every 7th column has a zero bias and holds EDGES"""
    gen = torch.Generator().manual_seed(seed)
    pre = torch.randn((B, N), generator=gen) * 6
    bias = torch.randn(N, generator=gen) * 0.5
    cols = torch.arange(0, N, 7)
    bias[cols] = 0.0
    edges = torch.tensor(EDGES, dtype=torch.float32)
    pre[:, cols] = edges[torch.arange(B * len(cols)) % len(edges)].reshape(B, len(cols))
    return pre, bias, gen


@pytest.mark.parametrize("N", [50, 257])
@pytest.mark.parametrize("act", ACTS)
def test_bias_act_matches_fp64(cuda_device, act, N):
    """act(pre + bias) within 4 ulp of fp64 on the fp32 pre-activation (softplus in the header's threshold form); the
    backward within 8 ulp of the reference's gradient, relative to the true value: relu g [y > 0], sigmoid g y (1 - y) on the
    kernel's output (TF SigmoidGrad), softplus g sigmoid(v) from the input (TF SoftplusGrad).  In place (out == pre,
    dpre == g) gives the same bits."""
    L = _lib.load()
    dev = cuda_device
    per_pass = elem_pass(dev)
    B = 2 * per_pass // N + 37
    assert B * N > 2 * per_pass
    pre, bias, gen = bias_act_inputs(B, N, seed=act * 1000 + N)
    pre_d, bias_d = pre.to(dev), bias.to(dev)

    out = nan_buffer((B, N), dev)
    call(L.mog_air_bias_act_forward, ptr(pre_d), ptr(bias_d), ptr(out), B, N, act)
    v = (pre + bias).double()                                       # one fp32 rounding, as in the kernel
    ref = {0: v, 1: v.clamp_min(0.0), 2: torch.where(v > 20, v, torch.log1p(torch.exp(v))), 3: torch.sigmoid(v)}[act]
    assert ulp_excess(out, ref, ref.abs(), 4) <= 1.0
    inplace = pre_d.clone()
    call(L.mog_air_bias_act_forward, ptr(inplace), ptr(bias_d), ptr(inplace), B, N, act)
    assert torch.equal(inplace, out)

    g = torch.randn((B, N), generator=gen)
    g_d = g.to(dev)
    dpre = nan_buffer((B, N), dev)
    call(L.mog_air_bias_act_backward, ptr(out), ptr(g_d), ptr(dpre), B * N, act)
    y, gg = f64(out), g.double()
    ref = {0: gg, 1: gg * (y > 0), 2: gg * torch.sigmoid(v), 3: gg * y * (1 - y)}[act]
    assert ulp_excess(dpre, ref, ref.abs(), 8) <= 1.0
    inplace = g_d.clone()
    call(L.mog_air_bias_act_backward, ptr(out), ptr(inplace), ptr(inplace), B * N, act)
    assert torch.equal(inplace, dpre)


@pytest.mark.parametrize("Ld", [50, 257])
def test_bias_gauss_matches_fp64(cuda_device, Ld):
    """mean and logvar bit-exact (one fp32 add each); latent within 4 ulp of the formula on the kernel's mean and logvar;
    the backward within 8 ulp of the sum of |terms| for each nullable gradient input alone and for all of them."""
    L = _lib.load()
    dev = cuda_device
    per_pass = elem_pass(dev)
    B = 2 * per_pass // Ld + 37
    assert B * Ld > 2 * per_pass
    gen = torch.Generator().manual_seed(Ld)
    pre = torch.randn((B, 2 * Ld), generator=gen)
    bm, bv = torch.randn(Ld, generator=gen) * 0.3, torch.randn(Ld, generator=gen) * 0.3
    eps = torch.randn((B, Ld), generator=gen)
    grads = {k: torch.randn((B, Ld), generator=gen) for k in ("g_mean", "g_logvar", "g_latent")}
    t = {k: v.to(dev) for k, v in dict(pre=pre, bm=bm, bv=bv, eps=eps, **grads).items()}

    mean, logvar, latent = (nan_buffer((B, Ld), dev) for _ in range(3))
    call(L.mog_air_bias_gauss_forward, ptr(t["pre"]), ptr(t["bm"]), ptr(t["bv"]), ptr(t["eps"]), ptr(mean), ptr(logvar), ptr(latent), B, Ld)
    assert torch.equal(mean.cpu(), pre[:, :Ld] + bm)
    assert torch.equal(logvar.cpu(), pre[:, Ld:] + bv)
    m, lv, e = f64(mean), f64(logvar), eps.double()
    noise = e * torch.exp(0.5 * lv)
    assert ulp_excess(latent, m + noise, m.abs() + noise.abs(), 4) <= 1.0

    half_sigma = 0.5 * torch.exp(0.5 * lv)
    for names in [("g_mean",), ("g_logvar",), ("g_latent",), ("g_mean", "g_logvar", "g_latent")]:
        g = {k: grads[k].double() if k in names else torch.zeros(B, Ld, dtype=torch.float64) for k in grads}
        dpre = nan_buffer((B, 2 * Ld), dev)
        call(L.mog_air_bias_gauss_backward, ptr(logvar), ptr(t["eps"]), *(ptr(t[k]) if k in names else None for k in grads), ptr(dpre),
             B, Ld)
        ref = torch.cat([g["g_mean"] + g["g_latent"], g["g_logvar"] + g["g_latent"] * e * half_sigma], 1)
        absterms = torch.cat([g["g_mean"].abs() + g["g_latent"].abs(), g["g_logvar"].abs() + (g["g_latent"] * e).abs() * half_sigma], 1)
        assert ulp_excess(dpre, ref, absterms, 8) <= 1.0, names


# ---------------------------------------------------------------------------------------------------------------------
# per-step elementwise kernels past one grid pass, under the bounds of tests/test_air_fused_gpu.py
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("act", [pytest.param(0, id="none"), pytest.param(1, id="tanh"), pytest.param(2, id="sigmoid")])
def test_gauss_sample_past_one_pass(cuda_device, act):
    L = _lib.load()
    dev = cuda_device
    per_pass = elem_pass(dev)
    n = 2 * per_pass + 12345
    assert n > 2 * per_pass
    gen = torch.Generator().manual_seed(20 + act)
    mean, lv, eps, gl, gs = (torch.randn(n, generator=gen) * s for s in (1.0, 0.7, 1.0, 1.0, 1.0))
    t = {k: v.to(dev) for k, v in dict(mean=mean, lv=lv, eps=eps, gl=gl, gs=gs).items()}

    latent = nan_buffer((n,), dev)
    squashed = nan_buffer((n,), dev) if act else None
    call(L.mog_air_gauss_sample_forward, ptr(t["mean"]), ptr(t["lv"]), ptr(t["eps"]), ptr(latent), ptr(squashed), n, act)
    m64, half_sigma = mean.double(), 0.5 * torch.exp(0.5 * lv.double())
    noise = eps.double() * 2 * half_sigma
    # relative to |mean| + |noise|: among this many draws some latents cancel to near 0, below the per-value bound's floor
    assert ulp_excess(latent, m64 + noise, m64.abs() + noise.abs(), 4) <= 1.0
    if act:                                                         # the squashing of the kernel's own latent
        ref = torch.tanh(f64(latent)) if act == 1 else torch.sigmoid(f64(latent))
        assert close_excess(squashed, ref, 2e-6, 1e-7) <= 1.0
        sq = f64(squashed)                                          # act' from the saved output, as TF's TanhGrad / SigmoidGrad
        dsq = 1 - sq * sq if act == 1 else sq * (1 - sq)

    for use_gl, use_gs in ((True, False), (False, True), (True, True)):
        d_mean, d_lv = nan_buffer((n,), dev), nan_buffer((n,), dev)
        call(L.mog_air_gauss_sample_backward, ptr(t["lv"]), ptr(t["eps"]), ptr(squashed), ptr(t["gl"]) if use_gl else None,
             ptr(t["gs"]) if use_gs else None, ptr(d_mean), ptr(d_lv), n, act)
        dl = torch.zeros(n, dtype=torch.float64)                   # g_squashed is ignored when act = 0
        if use_gl:
            dl = dl + gl.double()
        if use_gs and act:
            dl = dl + gs.double() * dsq
        assert close_excess(d_mean, dl, 1e-5, 1e-6) <= 1.0, (use_gl, use_gs)
        assert close_excess(d_lv, dl * eps.double() * half_sigma, 1e-5, 1e-6) <= 1.0, (use_gl, use_gs)


def test_thetas_past_one_pass(cuda_device):
    L = _lib.load()
    dev = cuda_device
    per_pass = elem_pass(dev)
    B = 2 * per_pass + 77
    assert B > 2 * per_pass
    gen = torch.Generator().manual_seed(30)
    shift = torch.tanh(torch.randn((B, 2), generator=gen))
    scale = torch.sigmoid(torch.randn(B, generator=gen) - 1)
    g_r, g_w = torch.randn((B, 6), generator=gen), torch.randn((B, 6), generator=gen)
    t = {k: v.to(dev) for k, v in dict(shift=shift, scale=scale, g_r=g_r, g_w=g_w).items()}

    th_r, th_w = nan_buffer((B, 6), dev), nan_buffer((B, 6), dev)
    call(L.mog_air_thetas_forward, ptr(t["shift"]), ptr(t["scale"]), ptr(th_r), ptr(th_w), B)
    s, x, y = scale, shift[:, 0], shift[:, 1]
    z = torch.zeros(B)
    assert torch.equal(th_r.cpu(), torch.stack([s, z, x, z, s, y], 1))                       # fp32 divides: the same bits
    assert torch.equal(th_w.cpu(), torch.stack([1 / s, z, -x / s, z, 1 / s, -y / s], 1))

    d_shift, d_scale = nan_buffer((B, 2), dev), nan_buffer((B,), dev)
    call(L.mog_air_thetas_backward, ptr(t["shift"]), ptr(t["scale"]), ptr(t["g_r"]), ptr(t["g_w"]), ptr(d_shift), ptr(d_scale), B)
    # GRAD_RTOL of the sum of |terms|: among this many draws, some small s make the 1 / s^2 terms of d_scale cancel
    s, x, y, gr, gw = s.double(), x.double(), y.double(), g_r.double(), g_w.double()
    ref_s = (gr[:, 0] + gr[:, 4]) - (gw[:, 0] + gw[:, 4]) / s ** 2 + (x * gw[:, 2] + y * gw[:, 5]) / s ** 2
    abs_s = (gr[:, 0].abs() + gr[:, 4].abs()) + (gw[:, 0].abs() + gw[:, 4].abs() + (x * gw[:, 2]).abs() + (y * gw[:, 5]).abs()) / s ** 2
    ref_xy = torch.stack([gr[:, 2] - gw[:, 2] / s, gr[:, 5] - gw[:, 5] / s], 1)
    abs_xy = torch.stack([gr[:, 2].abs() + gw[:, 2].abs() / s, gr[:, 5].abs() + gw[:, 5].abs() / s], 1)
    assert grad_excess(d_shift, ref_xy, abs_xy) <= 1.0
    assert grad_excess(d_scale, ref_s, abs_s) <= 1.0


@pytest.mark.parametrize("temp", [0.1, 1.0])
def test_zpres_past_one_pass(cuda_device, temp):
    L = _lib.load()
    dev = cuda_device
    per_pass = elem_pass(dev)
    B = 2 * per_pass + 77
    assert B > 2 * per_pass
    thr = 0.9
    gen = torch.Generator().manual_seed(40)
    lo = torch.randn(B, generator=gen) * 2
    u = torch.rand(B, generator=gen).clamp(1e-4, 1 - 1e-4)
    stop = torch.rand(B, generator=gen) * 1.5
    g_y, g_z = torch.randn(B, generator=gen), torch.randn(B, generator=gen)
    t = {k: v.to(dev) for k, v in dict(lo=lo, u=u, stop=stop, g_y=g_y, g_z=g_z).items()}

    y_pre, z_pres, stop_out = (nan_buffer((B,), dev) for _ in range(3))
    act_prev, act = (torch.full((B,), 0xAB, dtype=torch.uint8, device=dev) for _ in range(2))
    call(L.mog_air_zpres_forward, ptr(t["lo"]), ptr(t["u"]), ptr(t["stop"]), temp, thr, ptr(y_pre), ptr(z_pres), ptr(stop_out),
         ptr(act_prev), ptr(act), B)
    u64, s0 = u.double(), stop.double()
    ry = (lo.double() + torch.log(u64 + 1e-9) - torch.log(1 - u64 + 1e-9)) / temp
    rz = torch.sigmoid(ry)
    rs = s0 + 1 - rz
    assert close_excess(y_pre, ry, 1e-5, 1e-5) <= 1.0
    assert close_excess(z_pres, rz, 1e-5, 1e-6) <= 1.0
    z = f64(z_pres)
    assert close_excess(stop_out, s0 + (1 - z), 1e-6, 1e-6) <= 1.0    # the update of the kernel's own z_pres
    assert torch.equal(act_prev.cpu(), (stop < thr).to(torch.uint8))
    near = (rs - thr).abs() < 1e-5                                  # the mask may differ only on the threshold
    assert torch.equal(act.cpu()[~near], (rs < thr).to(torch.uint8)[~near])
    assert bool(((act.cpu() == 0) | (act.cpu() == 1)).all())

    # sigmoid' from the saved output z_pres, as TF's SigmoidGrad
    for use_y, use_z in ((True, False), (False, True), (True, True)):
        d_lo = nan_buffer((B,), dev)
        call(L.mog_air_zpres_backward, ptr(z_pres), ptr(t["g_y"]) if use_y else None, ptr(t["g_z"]) if use_z else None, temp,
             ptr(d_lo), B)
        ref = ((g_y.double() if use_y else 0.0) + (g_z.double() * z * (1 - z) if use_z else 0.0)) / temp
        assert close_excess(d_lo, ref, 1e-5, 1e-6) <= 1.0, (use_y, use_z)


@pytest.mark.parametrize("split", [False, True], ids=["gates", "gates+gates2"])
@pytest.mark.parametrize("B,Hh", [(4096, 256), (2389, 257)], ids=["4096x256", "2389x257"])
def test_lstm_pointwise_past_one_pass(cuda_device, B, Hh, split):
    """4096 x 256 is the LSTM of the C4 configuration (batch 4096)"""
    L = _lib.load()
    dev = cuda_device
    per_pass = elem_pass(dev)
    assert B * Hh > 2 * per_pass
    gen = torch.Generator().manual_seed(B + Hh + split)
    gates = torch.randn((B, 4 * Hh), generator=gen)
    gates2 = torch.randn((B, 4 * Hh), generator=gen) if split else None
    c_prev = torch.randn((B, Hh), generator=gen)
    g_h, g_c = torch.randn((B, Hh), generator=gen), torch.randn((B, Hh), generator=gen)
    t = {k: to_dev(v, dev) for k, v in dict(gates=gates, gates2=gates2, c_prev=c_prev, g_h=g_h, g_c=g_c).items()}

    c_new, h_new = nan_buffer((B, Hh), dev), nan_buffer((B, Hh), dev)
    call(L.mog_air_lstm_pointwise_forward, ptr(t["gates"]), ptr(t["gates2"]), ptr(t["c_prev"]), ptr(c_new), ptr(h_new), B, Hh)
    total = (gates.double() + (gates2.double() if split else 0.0)).requires_grad_(True)
    c64 = c_prev.double().requires_grad_(True)
    i, j, f, o = total.chunk(4, 1)                                  # tf.nn.rnn_cell.LSTMCell, forget_bias = 1
    rc = torch.sigmoid(f + 1.0) * c64 + torch.sigmoid(i) * torch.tanh(j)
    rh = torch.sigmoid(o) * torch.tanh(rc)
    assert close_excess(c_new, rc.detach(), 1e-5, 1e-6) <= 1.0
    assert close_excess(h_new, rh.detach(), 1e-5, 1e-6) <= 1.0

    for use_h, use_c in ((True, True), (True, False), (False, True)):
        d_gates, d_c_prev = nan_buffer((B, 4 * Hh), dev), nan_buffer((B, Hh), dev)
        call(L.mog_air_lstm_pointwise_backward, ptr(t["gates"]), ptr(t["gates2"]), ptr(t["c_prev"]), ptr(c_new),
             ptr(t["g_h"]) if use_h else None, ptr(t["g_c"]) if use_c else None, ptr(d_gates), ptr(d_c_prev), B, Hh)
        loss = (rh * g_h.double()).sum() if use_h else 0.0
        if use_c:
            loss = loss + (rc * g_c.double()).sum()
        rg, rcp = torch.autograd.grad(loss, (total, c64), retain_graph=True)
        assert close_excess(d_gates, rg, 1e-5, 1e-6) <= 1.0, (use_h, use_c)
        assert close_excess(d_c_prev, rcp, 1e-5, 1e-6) <= 1.0, (use_h, use_c)


# ---------------------------------------------------------------------------------------------------------------------
# reconstruction loss: mog_bce_recon_* past one grid pass
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("P", [2500, 2501])
def test_bce_recon_past_one_pass(cuda_device, P):
    """P = 2500: every row 16-byte aligned (float4 path); P = 2501: every fourth row, so rows mix the float4 and scalar paths.
    Bounds of tests/test_bce_gpu.py against oracle/bce_ref.py; mse = NULL leaves the loss unchanged."""
    L = _lib.load()
    dev = cuda_device
    fwd_pass, bwd_pass = bce_fwd_pass(dev), bce_bwd_pass(dev)
    B = fwd_pass + fwd_pass // 2 + 3
    assert B > fwd_pass and B > 2 * bwd_pass
    rng = np.random.default_rng(P)
    # canvases like running_recon: many exact zeros, values above 1 where windows overlap, a few negatives
    c = rng.random((B, P), dtype=np.float32) * 1.4 - 0.1
    c[rng.random((B, P), dtype=np.float32) < 0.5] = 0.0
    c[rng.random((B, P), dtype=np.float32) < 0.01] = 1.0
    x = np.clip(rng.random((B, P), dtype=np.float32) * 1.2, 0, 1).astype(np.float32)
    x[rng.random((B, P), dtype=np.float32) < 0.6] = 0.0
    g = rng.normal(size=B).astype(np.float32)
    cd, xd, gd = (torch.from_numpy(a).to(dev) for a in (c, x, g))

    loss, mse = nan_buffer((B,), dev), nan_buffer((B,), dev)
    call(L.mog_bce_recon_forward, ptr(cd), ptr(xd), ptr(loss), ptr(mse), B, P)
    ref_loss, ref_mse = bce_ref.reconstruction_loss(c, x)
    mag = bce_ref.term_magnitudes(c, x)
    assert np.all(np.abs(loss.cpu().numpy() - ref_loss) <= 2e-6 * mag + 1e-12)
    np.testing.assert_allclose(mse.cpu().numpy(), ref_mse, rtol=2e-6, atol=1e-12)
    loss_only = nan_buffer((B,), dev)
    call(L.mog_bce_recon_forward, ptr(cd), ptr(xd), ptr(loss_only), None, B, P)
    assert torch.equal(loss_only, loss)

    dcanvas = nan_buffer((B, P), dev)
    call(L.mog_bce_recon_backward, ptr(cd), ptr(xd), ptr(gd), ptr(dcanvas), B, P)
    got = dcanvas.cpu().numpy()
    ref = bce_ref.reconstruction_loss_backward(c, x, g)
    r = np.clip(c.astype(np.float64), 0, 1)
    dmag = (np.abs(x / (r + 1e-10)) + np.abs((1 - x) / (1 - r + 1e-10))) * np.abs(g)[:, None]   # the two terms may cancel
    assert np.all(got[(c < 0) | (c > 1)] == 0)                     # the clip mask (inclusive bounds) is exact
    assert np.all(np.abs(got - ref) <= 2e-6 * dmag + 1e-30)


# ---------------------------------------------------------------------------------------------------------------------
# KL terms of the ELBO: mog_air_kl_forward / _backward
# ---------------------------------------------------------------------------------------------------------------------
# One thread per image, ceil(B / 128) CTAs and no grid-stride loop: B = 127, 128, 129 sit around the CTA boundary and
# 4097 leaves one thread in the last CTA.  T = 1 ... 16 steps, L = 1, 50 (the model's) and 257 VAE latents.
KL_SHAPES = [pytest.param(1, 1, 1, id="B1-T1-L1"), pytest.param(127, 2, 50, id="B127-T2-L50"),
             pytest.param(128, 16, 1, id="B128-T16-L1"), pytest.param(129, 6, 257, id="B129-T6-L257"),
             pytest.param(129, 16, 50, id="B129-T16-L50"), pytest.param(4097, 6, 50, id="B4097-T6-L50"),
             pytest.param(4097, 1, 257, id="B4097-T1-L257")]
# the model's priors (AIRConfig): scale N(-1, 0.05), VAE N(0, 1) -- mean, variance, mean, variance
KL_PRIORS = (-1.0, 0.05, 0.0, 1.0)
KL_INPUTS = ("y_pre", "prior_lo", "post_lo", "active_prev", "active", "sc_mean", "sc_lv", "sh_mean", "sh_lv", "g_sh_mean",
             "g_sh_lv", "v_mean", "v_lv")
KL_GRADS = tuple(k for k in KL_INPUTS if not k.startswith("active"))   # d_<name>, in the order of the C ABI
CONCRETE = ("y_pre", "prior_lo", "post_lo")
SHIFT = ("sh_mean", "sh_lv", "g_sh_mean", "g_sh_lv")
# what image b is for, by b % 8: 0, 6, 7 general; 1 post_lo == prior_lo at every step; 2 shift posterior == learned
# prior at every step; 3 g_kl = 0; 4 every step masked; 5 log-variances out to +-80
ROLE_SAME_LO, ROLE_SAME_SHIFT, ROLE_NO_GRAD, ROLE_MASKED, ROLE_WIDE_LV = 1, 2, 3, 4, 5


def kl_inputs(B, T, L, temp, seed):
    """fp32 [T][B][..] stacks.  Log-odds up to +-30 with y_pre the posterior's Concrete logit (log-odds plus logistic
    noise, over the temperature); about 10 % of the steps planted so that a = -y temp + l (prior or posterior) lies near
    +-50, +-89 or +-100, past where expf overflows.  Log-variances stay within +-80 and the shift's within what its
    ratio exp(lv - glv) and dm^2 / exp(glv) keep finite: above about 88.7 expf(lv) overflows and a masked step's
    gradient becomes 0 * inf = NaN, as in the framework form -- outside the contract, not tested."""
    rng = np.random.default_rng(seed)
    role = np.arange(B) % 8
    lq, lp = rng.uniform(-30, 30, (T, B)), rng.uniform(-30, 30, (T, B))
    u = rng.uniform(1e-4, 1 - 1e-4, (T, B))
    y = (lq + np.log(u) - np.log1p(-u)) / temp
    planted = rng.random((T, B)) < 0.1
    edge = rng.choice([-100.0, -89.0, -50.0, 50.0, 89.0, 100.0], (3, T, B))
    at_zero_y = planted & (rng.random((T, B)) < 0.5)             # y = 0: a = l on both sides
    y[at_zero_y], lp[at_zero_y], lq[at_zero_y] = 0.0, edge[0][at_zero_y], edge[1][at_zero_y]
    from_y = planted & ~at_zero_y                                # y = -a / temp: a = edge + l, with |l| <= 30
    y[from_y] = -edge[2][from_y] / temp
    lp[:, role == ROLE_SAME_LO] = lq[:, role == ROLE_SAME_LO]
    x = {"y_pre": y, "prior_lo": lp, "post_lo": lq,
         "sc_mean": rng.normal(-1, 2, (T, B)), "sc_lv": rng.normal(0, 1.5, (T, B)),
         "sh_mean": rng.normal(0, 1, (T, B, 2)), "sh_lv": rng.normal(0, 1.5, (T, B, 2)),
         "g_sh_mean": rng.normal(0, 1, (T, B, 2)), "g_sh_lv": rng.normal(0, 1.5, (T, B, 2)),
         "v_mean": rng.normal(0, 2, (T, B, L)), "v_lv": rng.normal(0, 1.5, (T, B, L))}
    wide = role == ROLE_WIDE_LV
    for k in ("sc_lv", "v_lv", "sh_lv"):
        v = rng.uniform(-80, 80, x[k][:, wide].shape)
        v.reshape(-1)[::5] = rng.choice([-80.0, 80.0], v.reshape(-1)[::5].shape)
        x[k][:, wide] = v
    lv = x["sh_lv"][:, wide]
    x["g_sh_lv"][:, wide] = rng.uniform(np.maximum(-80.0, lv - 80.0), 80.0)      # lv - glv <= 80
    for k in ("sh_mean", "sh_lv"):
        x["g_" + k][:, role == ROLE_SAME_SHIFT] = x[k][:, role == ROLE_SAME_SHIFT]
    x = {k: v.astype(np.float32) for k, v in x.items()}
    combo = rng.integers(0, 4, (T, B))                           # (active_prev, active) = (combo & 1, combo >> 1)
    combo[0, :min(B, 4)] = np.arange(min(B, 4))                  # every combination, active without active_prev included
    combo[:, role == ROLE_MASKED] = 0
    x["active_prev"], x["active"] = (combo & 1).astype(np.uint8), (combo >> 1).astype(np.uint8)
    g = rng.normal(0, 1, B).astype(np.float32)
    g[role == ROLE_NO_GRAD] = 0.0
    return x, g, role


def kl_reference(x, g, temp, priors):
    """The header's formulas in fp64 on the fp32 inputs and constants: per image the four components and kl, the closed-form
    gradients, and for each the sum of |terms| entering it.  The Concrete term's |terms| include the shared
    |log_temp| + |y (temp + 1)| that cancels between posterior and prior, and for every use of a = -y temp + l the
    magnitude |y temp| + |l| of the fp32 a (its rounding moves lse0 by up to sigma(a) and sigma by sigma (1 - sigma) times
    that)."""
    tf, spm, spv, vpm, vpv = (float(np.float32(v)) for v in (temp,) + tuple(priors))
    d = {k: v.astype(np.float64) for k, v in x.items()}
    y, lp, lq, mp, m = d["y_pre"], d["prior_lo"], d["post_lo"], d["active_prev"], d["active"]
    g = g.astype(np.float64)
    gz, gm = mp * g, m * g
    r, A = {}, {}

    lt = np.log(tf + 1e-9)
    ap, aq = -y * tf + lp, -y * tf + lq
    cp, cq = np.abs(y * tf) + np.abs(lp), np.abs(y * tf) + np.abs(lq)
    log_density = lambda l, a: lt - y * (tf + 1) + l - 2 * np.logaddexp(0, a)   # air/concrete.py:30-64
    z = log_density(lq, aq) - log_density(lp, ap)
    Az = (2 * (abs(lt) + np.abs(y * (tf + 1))) + np.abs(lp) + np.abs(lq) + 2 * (np.logaddexp(0, ap) + np.logaddexp(0, aq))
          + 2 * (cp + cq))
    sp, sq = special.expit(ap), special.expit(aq)
    r["y_pre"], A["y_pre"] = gz * 2 * tf * (sq - sp), np.abs(gz) * 2 * tf * (sq + sp + sq * (1 - sq) * cq + sp * (1 - sp) * cp)
    r["post_lo"], A["post_lo"] = gz * (1 - 2 * sq), np.abs(gz) * (1 + 2 * sq + 2 * sq * (1 - sq) * cq)
    r["prior_lo"], A["prior_lo"] = -gz * (1 - 2 * sp), np.abs(gz) * (1 + 2 * sp + 2 * sp * (1 - sp) * cp)

    def fixed_prior(name, gm, pm, pv):                           # scale and VAE latents: :731-736, :769-774
        mu, lv = d[name + "_mean"], d[name + "_lv"]
        ev, dm, am = np.exp(lv), mu - pm, np.abs(mu) + abs(pm)
        kl = 0.5 * (np.log(pv) - lv - 1 + ev / pv + dm * dm / pv)
        Akl = 0.5 * (abs(np.log(pv)) + np.abs(lv) + 1 + ev / pv + am * am / pv)
        r[name + "_mean"], A[name + "_mean"] = gm * dm / pv, np.abs(gm) * am / pv
        r[name + "_lv"], A[name + "_lv"] = gm * 0.5 * (ev / pv - 1), np.abs(gm) * 0.5 * (ev / pv + 1)
        return kl, Akl

    ksc, Asc = fixed_prior("sc", gm, spm, spv)
    kv, Av = fixed_prior("v", gm[..., None], vpm, vpv)
    mu, lv, gmu, glv = d["sh_mean"], d["sh_lv"], d["g_sh_mean"], d["g_sh_lv"]   # shift, learned prior: :750-755
    ratio, inv_gvar, dm, am, gm2 = np.exp(lv - glv), np.exp(-glv), mu - gmu, np.abs(mu) + np.abs(gmu), gm[..., None]
    ksh = 0.5 * (glv - lv - 1 + ratio + dm * dm * inv_gvar)
    Ash = 0.5 * (np.abs(glv) + np.abs(lv) + 1 + ratio + am * am * inv_gvar)
    r["sh_mean"], A["sh_mean"] = gm2 * dm * inv_gvar, np.abs(gm2) * am * inv_gvar
    r["g_sh_mean"], A["g_sh_mean"] = -r["sh_mean"], A["sh_mean"]
    r["sh_lv"], A["sh_lv"] = gm2 * 0.5 * (ratio - 1), np.abs(gm2) * 0.5 * (ratio + 1)
    r["g_sh_lv"] = gm2 * 0.5 * (1 - ratio - dm * dm * inv_gvar)
    A["g_sh_lv"] = np.abs(gm2) * 0.5 * (1 + ratio + am * am * inv_gvar)

    comps = np.stack([(mp * z).sum(0), (m * ksc).sum(0), (m * ksh.sum(-1)).sum(0), (m * kv.sum(-1)).sum(0)], 1)
    Acomps = np.stack([(mp * Az).sum(0), (m * Asc).sum(0), (m * Ash.sum(-1)).sum(0), (m * Av.sum(-1)).sum(0)], 1)
    return comps, Acomps, r, A


def np_excess(got, ref, mag, ulps, floor=FLT_MIN):
    """ulp_excess on numpy arrays: max of |got - ref| / (ulps * 2^-23 * mag + floor); <= 1 passes, a NaN in got fails"""
    err = np.abs(np.asarray(got, np.float64) - ref) / (ulps * EPS32 * mag + floor)
    return float(np.nan_to_num(err, nan=np.inf).max())


@pytest.mark.parametrize("temp", [0.1, 1.0])
@pytest.mark.parametrize("B,T,Ld", KL_SHAPES)
def test_kl_matches_fp64(cuda_device, B, T, Ld, temp):
    """mog_air_kl_forward / _backward against the fp64 formulas, every output NaN-filled first.
    Forward: each component within 4 ulp x summation depth x sum of |terms| (the depth of its running sum over steps,
    and latents, plus the few roundings of one term); kl likewise with three more additions.  This bound is the
    contract: the forward value feeds only the loss value, not the gradients, so the Concrete term keeps the reference's
    form (air/concrete.py), in which the shared log_temp - y (temp + 1) cancels.  kl is ((c0 + c1) + c2) + c3 in fp32 bit
    for bit, the same bits without components; a component is exactly 0 where its mask is off at every step, c0 where
    post_lo == prior_lo, c2 where the shift posterior equals its learned prior.
    Backward: every d_* within 8 ulp of the sum of |terms| of its closed form, exactly 0 (either sign) at masked steps, in
    g_kl = 0 images, for d_y_pre where post_lo == prior_lo and for the four shift gradients where the posterior equals the
    prior.  The two masks are applied independently: active_prev gates the Concrete term, active the other three."""
    L = _lib.load()
    dev = cuda_device
    x, g, role = kl_inputs(B, T, Ld, temp, seed=B * 1000 + T * 10 + Ld + int(temp * 7))
    t = {k: torch.from_numpy(v).to(dev) for k, v in x.items()}
    g_d = torch.from_numpy(g).to(dev)
    ins = [ptr(t[k]) for k in KL_INPUTS]
    comps_ref, Acomps, r, A = kl_reference(x, g, temp, KL_PRIORS)
    mp, m = x["active_prev"].astype(bool), x["active"].astype(bool)
    assert B < 4 or len(set(zip(mp[0, :4], m[0, :4]))) == 4

    kl, comps = nan_buffer((B,), dev), nan_buffer((B, 4), dev)
    call(L.mog_air_kl_forward, *ins, B, T, Ld, temp, *KL_PRIORS, ptr(kl), ptr(comps))
    kl_only = nan_buffer((B,), dev)
    call(L.mog_air_kl_forward, *ins, B, T, Ld, temp, *KL_PRIORS, ptr(kl_only), None)
    kl, comps, kl_only = kl.cpu().numpy(), comps.cpu().numpy(), kl_only.cpu().numpy()
    assert np.array_equal(kl_only.view(np.uint32), kl.view(np.uint32))
    summed = ((comps[:, 0] + comps[:, 1]) + comps[:, 2]) + comps[:, 3]          # fp32 additions, in the kernel's order
    assert np.array_equal(summed.view(np.uint32), kl.view(np.uint32))
    depth = np.array([T + 8, T + 8, 2 * T + 8, T * Ld + 8])
    for i in range(4):
        assert np_excess(comps[:, i], comps_ref[:, i], depth[i] * Acomps[:, i], 4) <= 1.0, i
    assert np_excess(kl, comps_ref.sum(1), (depth.max() + 3) * Acomps.sum(1), 4) <= 1.0
    assert np.all(comps[~mp.any(0), 0] == 0) and np.all(comps[~m.any(0), 1:] == 0)
    assert np.all(kl[role == ROLE_MASKED] == 0)
    assert np.all(comps[role == ROLE_SAME_LO, 0] == 0)
    assert np.all(comps[role == ROLE_SAME_SHIFT, 2] == 0)

    d = {k: nan_buffer(x[k].shape, dev) for k in KL_GRADS}
    call(L.mog_air_kl_backward, *ins, B, T, Ld, temp, *KL_PRIORS, ptr(g_d), *(ptr(d[k]) for k in KL_GRADS))
    d = {k: v.cpu().numpy() for k, v in d.items()}
    # below a ~ -88.7, expf(-a) overflows and sigm(a) is 0 where the true value is a denormal below FLT_MIN: d_y_pre carries
    # that absolute error times 2 temp |g|
    floor = {"y_pre": FLT_MIN * (1 + 4 * float(np.float32(temp)) * np.abs(g))}
    for k in KL_GRADS:
        assert np_excess(d[k], r[k], A[k], 8, floor.get(k, FLT_MIN)) <= 1.0, k
        on = mp if k in CONCRETE else m                          # the step's own mask, not the other one
        off = ~on[(...,) + (None,) * (d[k].ndim - 2)] | (g == 0)[(slice(None),) + (None,) * (d[k].ndim - 2)]
        assert np.all(d[k][np.broadcast_to(off, d[k].shape)] == 0), k
    assert np.all(d["y_pre"][:, role == ROLE_SAME_LO] == 0)
    assert np.array_equal(d["prior_lo"][:, role == ROLE_SAME_LO], -d["post_lo"][:, role == ROLE_SAME_LO])
    for k in SHIFT:
        assert np.all(d[k][:, role == ROLE_SAME_SHIFT] == 0), k
