"""CPU tests of the drop-in boundary: libmogstn.so loads, exports every symbol include/mogstn.h declares,
and validates arguments before touching the device (no compute calls here)."""
import ctypes
import os
import re

import pytest

from mog_asr_b200 import _lib, build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    build.build()
    return _lib.load()


def header_symbols():
    text = open(os.path.join(ROOT, "include", "mogstn.h")).read()
    return re.findall(r"MOG_API\s+(?:int|size_t)\s+(mog_[a-z_]+)\s*\(", text)


def test_every_declared_symbol_is_exported_and_bound(lib):
    names = header_symbols()
    assert len(names) >= 10
    raw = ctypes.CDLL(_lib.SO_PATH)
    for n in names:
        assert hasattr(raw, n), f"{n} declared in mogstn.h but not exported"
    assert sorted(names) == sorted(_lib.SIGNATURES), "ctypes binding and header disagree"
    assert lib.mog_version() == _lib.ABI_VERSION


def test_asr_config_struct_layout_matches_header():
    # 3 scalars + 8 counts + 8 floats, all 4-byte: 76 bytes, no padding
    assert ctypes.sizeof(_lib.AsrConfig) == 4 * (3 + _lib.MOG_ASR_MAX_COUNTS + 8)
    text = open(os.path.join(ROOT, "include", "mogstn.h")).read()
    assert f"#define MOG_ASR_MAX_COUNTS {_lib.MOG_ASR_MAX_COUNTS}" in text
    assert f"#define MOG_ASR_MAX_STEPS {_lib.MOG_ASR_MAX_STEPS}" in text


def test_bad_arguments_are_rejected_before_any_launch(lib):
    one = 0x1000  # never dereferenced: validation fails first
    assert lib.mog_stn_forward(one, one, one, 4, 0, 50, 1, 28, 28, 1, None) == -2        # MOG_ERR_DIM
    assert "non-positive" in _lib.last_error()
    assert lib.mog_stn_forward(one, one, one, 5, 50, 50, 1, 28, 28, 2, None) == -2       # u_batch_div must divide B
    assert lib.mog_stn_forward(None, one, one, 4, 50, 50, 1, 28, 28, 1, None) == -1      # MOG_ERR_NULL
    assert lib.mog_stn_forward(one, one, one, 4, 1 << 15, 1 << 15, 1, 28, 28, 1, None) == -3   # MOG_ERR_OVERFLOW
    assert lib.mog_stn_backward(one, one, None, one, one, 4, 50, 50, 1, 28, 28, 1, None) == -1
    assert lib.mog_stn_corners(None, one, 4, 50, 50, 28, 28, None) == -1
    cfg = _lib.AsrConfig()
    assert lib.mog_asr_reg_forward(one, one, one, None, 1.0, 4, 99, ctypes.byref(cfg), one, None, one, None) == -2
    with pytest.raises(RuntimeError, match="bad argument"):
        _lib.check(lib.mog_stn_forward(one, one, one, 4, 0, 50, 1, 28, 28, 1, None), "mog_stn_forward")
    # the rows built around the sampler validate the same way
    assert lib.mog_detection_eval(one, one, one, one, one, one, 4, 9, 3, 50.0, one, one, one, one, one, None) == -2   # > 8 boxes
    assert "max 8 boxes" in _lib.last_error()
    assert lib.mog_detection_eval(one, one, None, one, one, one, 4, 3, 3, 50.0, one, one, one, one, one, None) == -1
    counts = (ctypes.c_int * 2)(1, 3)
    assert lib.mog_synth_place(1, 0, 4, 50, 3, counts, 2, 17, 23, 0, 0, 2, 0, 8, one, one, one, one, None) == -2      # mode 2
    assert lib.mog_synth_place(1, 0, 4, 50, 2, counts, 2, 17, 23, 0, 0, 0, 0, 8, one, one, one, one, None) == -2      # count 3 > max_objects 2
    assert "exceeds max_objects" in _lib.last_error()
    assert lib.mog_synth_place(1, 0, 4, 50, 3, counts, 2, 17, 23, 0, 0, 0, 0, 8, None, one, one, one, None) == -1
    assert lib.mog_bce_recon_forward(one, one, one, None, 4, 0, None) == -2

    # KL terms: 13 inputs, B, T, L, temperature, scale prior mean / variance, VAE prior mean / variance, then the outputs
    def kl_forward(B=4, T=3, L=50, temp=0.1, spv=0.05, vpv=1.0, inputs=(one,) * 13, kl=one):
        return lib.mog_air_kl_forward(*inputs, B, T, L, temp, -1.0, spv, 0.0, vpv, kl, None, None)

    def kl_backward(B=4, T=3, L=50, temp=0.1, spv=0.05, vpv=1.0, inputs=(one,) * 13, outs=(one,) * 12):
        return lib.mog_air_kl_backward(*inputs, B, T, L, temp, -1.0, spv, 0.0, vpv, *outs, None)   # g_kl, then 11 d_*

    for fn in (kl_forward, kl_backward):
        for bad in (dict(B=-1), dict(T=0), dict(L=0), dict(temp=0.0), dict(temp=-0.1), dict(spv=0.0), dict(vpv=-1.0)):
            assert fn(**bad) == -2, (fn.__name__, bad)
        for i in range(13):
            assert fn(inputs=(one,) * i + (None,) + (one,) * (12 - i)) == -1, (fn.__name__, i)
    assert kl_forward(kl=None) == -1
    for i in range(12):
        assert kl_backward(outs=(one,) * i + (None,) + (one,) * (11 - i)) == -1, i


def test_zero_batch_is_a_no_op(lib):
    assert lib.mog_stn_forward(None, None, None, 0, 50, 50, 1, 28, 28, 1, None) == 0
    assert lib.mog_stn_backward(None, None, None, None, None, 0, 50, 50, 1, 28, 28, 1, None) == 0
    assert lib.mog_detection_eval(None, None, None, None, None, None, 0, 3, 3, 50.0, None, None, None, None, None, None) == 0
    assert lib.mog_synth_place(1, 0, 0, 50, 3, (ctypes.c_int * 1)(1), 1, 17, 23, 0, 0, 0, 0, 8, None, None, None, None, None) == 0
    assert lib.mog_air_kl_forward(*(None,) * 13, 0, 3, 50, 0.1, -1.0, 0.05, 0.0, 1.0, None, None, None) == 0
    assert lib.mog_air_kl_backward(*(None,) * 13, 0, 3, 50, 0.1, -1.0, 0.05, 0.0, 1.0, *(None,) * 12, None) == 0


def test_host_wrappers_refuse_cpu_tensors():
    import torch
    import mog_asr_b200 as m
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m.transformer(torch.zeros(1, 4, 4, 1), torch.zeros(1, 6), (2, 2))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m.write_composite(torch.zeros(1, 4, 4), torch.zeros(1, 2, 2), torch.zeros(1, 6), torch.zeros(1))
    from mog_asr_b200.host_api import HostCompositeWriter, HostSampler
    from mog_asr_b200.sxy import read_glimpse_sxy, write_composite_sxy
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        read_glimpse_sxy(torch.zeros(1, 4, 4, 1), torch.zeros(1, 2), torch.ones(1), (2, 2))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        write_composite_sxy(torch.zeros(1, 4, 4), torch.zeros(1, 2, 2), torch.zeros(1, 2), torch.ones(1), torch.zeros(1))
    for ctor in (lambda: HostSampler("cpu", (4, 4), (2, 2)), lambda: HostCompositeWriter("cpu", (2, 2), (4, 4), steps=2)):
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            ctor()


def test_zero_batch_is_a_no_op_for_the_newer_entry_points(lib):
    """argument checks and the B = 0 early-outs run on the host: no GPU needed"""
    assert lib.mog_stn_read_sxy_forward(None, None, None, None, 0, 50, 50, 28, 28, None) == 0
    assert lib.mog_stn_read_sxy_backward(None, None, None, None, None, None, None, None, None, 0, 50, 50, 28, 28, None) == 0
    assert lib.mog_stn_write_composite_sxy_forward(None, None, None, None, None, 0.9, None, None, 0, 28, 28, 50, 50, None) == 0
    assert lib.mog_stn_write_composite_sxy_backward(None, None, None, None, None, 0.9, None, None, None, None, None, None, None,
                                                    0, 28, 28, 50, 50, None) == 0
    assert lib.mog_stn_write_composite_host(None, None, None, None, None, None, None, None, 0, 8, 28, 28, 50, 50, 64, None, 0, None, 3) == 0
    assert lib.mog_stn_write_composite_host_workspace_bytes(64, 8, 28, 28, 50, 50, 3) > 0
    assert lib.mog_stn_write_composite_host_workspace_bytes(0, 8, 28, 28, 50, 50, 3) == 0
    assert lib.mog_stn_read_sxy_forward(None, None, None, None, 4, 50, 50, 28, 28, None) < 0        # NULL pointers with B > 0
    assert lib.mog_stn_read_sxy_forward(None, None, None, None, 4, 0, 50, 28, 28, None) < 0         # bad dimension


def test_product_package_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "mog_asr_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, re.M), f"{f} imports the oracle"
                assert "libstnref" not in src, f"{f} references the oracle library"
