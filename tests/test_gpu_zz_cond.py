"""Conditioning producer on the device (SURVEY.md 8f next-2): nvwn_set_conditioning_from_features must leave the
engine in exactly the state nvwn_set_inputs(Lh) leaves it in when Lh is the host restatement of the same arithmetic
(itself checked against the reference's module in tests/test_cond_producer.py): identical sampled indices."""
import ctypes as C
import os

import numpy as np
import pytest

from tests import refgen
from tests.test_cond_producer import GOLD, golden_lh, host_cond

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("dtype_name", ["fp32", "fp16"])
def test_generation_from_features_equals_generation_from_host_conditioning(dtype_name):
    import nv_wavenet_b200 as nw
    rng = np.random.default_rng(5)
    L, R, S, A, md = 4, 64, 256, 256, 4
    B, Cc, T, window, stride = 3, 6, 5, 24, 8                    # 40 samples
    N = T * stride + 6                                           # the producer fills [6, 46)
    first = 6
    w = refgen.lively_inputs(31, R, S, A, L, B, N)
    g = {"x_features": rng.standard_normal((B, Cc, T)).astype(np.float32),
         "x_upsample_weight": (0.3 * rng.standard_normal((Cc, Cc, window))).astype(np.float32),
         "x_upsample_bias": (0.1 * rng.standard_normal(Cc)).astype(np.float32),
         "x_cond_weight": (np.abs(w["Lh"]).max() * rng.standard_normal((L * 2 * R, Cc))).astype(np.float32),
         "x_cond_bias": (0.1 * np.abs(w["Lh"]).max() * rng.standard_normal(L * 2 * R)).astype(np.float32),
         "x_geometry": np.array([Cc, T, window, stride, L, R, B])}
    lh = np.array(w["Lh"], np.float32)                           # [N][L][B][2R]; samples before `first` keep the synthetic values
    lh[first:] = host_cond(g, "x")

    dt = nw.FP16 if dtype_name == "fp16" else nw.FP32
    ys = []
    for mode in ("host", "device"):
        e = nw.NVWavenetInfer(L, md, B, N, R=R, S=S, A=A, dtype=dt)
        e.load(w)
        if mode == "host":
            e.set_inputs(lh, w["selectors"])
        else:
            e.set_inputs(np.ascontiguousarray(w["Lh"], np.float32), w["selectors"])
            n = e.set_conditioning_from_features(g["x_features"], g["x_upsample_weight"], g["x_upsample_bias"], g["x_cond_weight"],
                                                 g["x_cond_bias"], stride, first_sample=first)
            assert n == T * stride
        y = np.zeros((B, N), np.int32)
        e.run(N, B, y); e.synchronize()
        ys.append(y)
    assert np.array_equal(ys[0], ys[1])
    assert len(np.unique(ys[0])) > 2


@pytest.mark.parametrize("kernel", ["fp32", "stream", "tc", "lat"])
def test_device_conditioning_store_matches_reference_module(kernel, monkeypatch):
    """The tensor the device producer leaves in the engine's conditioning store (read back through a debug getter, whatever the
    kernel-native layout) against vectors from the reference's own WaveNet.get_cond_input (tests/golden/make_golden_cond.py):
    fp32 within 1e-5 of the tensor scale, fp16 stores within 1e-3."""
    import nv_wavenet_b200 as nw
    from nv_wavenet_b200 import _lib
    for k in ("NVWN_FP16_KERNEL", "NVWN_TC_TILE", "NVWN_TC_NODUP"):
        monkeypatch.delenv(k, raising=False)
    if kernel != "fp32":
        monkeypatch.setenv("NVWN_FP16_KERNEL", kernel)
    Cc, T, window, stride, L, R, B = [int(v) for v in GOLD["c_geometry"]]
    N = T * stride + 5
    first = 5
    e = nw.NVWavenetInfer(L, 2, B, N, R=R, S=256, A=256, dtype=nw.FP32 if kernel == "fp32" else nw.FP16)
    n = e.set_conditioning_from_features(GOLD["c_features"], GOLD["c_upsample_weight"], GOLD["c_upsample_bias"], GOLD["c_cond_weight"],
                                         GOLD["c_cond_bias"], stride, first_sample=first)
    assert n == T * stride
    lib = _lib.lib()
    lib.nvwn_debug_get_conditioning.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int]
    full = np.full((n, L, B, 2 * R), np.nan, np.float32)
    assert lib.nvwn_debug_get_conditioning(e._h, C.c_void_p(full.ctypes.data), first, n) == 0
    got, want = golden_lh(full, "c")
    scale = np.abs(want).max()
    tol = 1e-5 if kernel == "fp32" else 1e-3
    assert np.isfinite(full).all() and np.abs(got - want).max() <= tol * scale, np.abs(got - want).max() / scale


def test_out_of_range_is_rejected():
    import nv_wavenet_b200 as nw
    e = nw.NVWavenetInfer(2, 2, 2, 16, R=64, S=256, A=256, dtype=nw.FP32)
    z = np.zeros((2, 3, 5), np.float32)
    with pytest.raises(Exception):
        e.set_conditioning_from_features(z, np.zeros((3, 3, 8), np.float32), np.zeros(3, np.float32), np.zeros((2 * 2 * 64, 3), np.float32),
                                         np.zeros(2 * 2 * 64, np.float32), 4)        # 5 * 4 = 20 samples > 16


def test_producer_ranges_on_a_side_stream_equal_the_one_shot_call_and_the_host_arithmetic():
    """nvwn_cond_producer_load + _run over three unequal sample ranges on a second stream (the overlapped pipeline of bench.py) must
    leave the same store as the one-shot call; and the fp32 store must equal the host restatement of the same arithmetic BIT FOR BIT
    (the register-tiled projection kernel keeps the element function's accumulation order).  Shape: two ragged 128-row tiles, odd L."""
    import torch
    import nv_wavenet_b200 as nw
    from nv_wavenet_b200 import _lib
    rng = np.random.default_rng(11)
    L, R, B = 5, 64, 19
    Cc, T, window, stride = 80, 7, 32, 8                         # 56 samples: 56 x 19 = 1064 rows = 8 full + 1 ragged 128-row tile
    N = T * stride + 3
    first = 3
    g = {"x_features": rng.standard_normal((B, Cc, T)).astype(np.float32),
         "x_upsample_weight": (0.1 * rng.standard_normal((Cc, Cc, window))).astype(np.float32),
         "x_upsample_bias": (0.1 * rng.standard_normal(Cc)).astype(np.float32),
         "x_cond_weight": (0.1 * rng.standard_normal((L * 2 * R, Cc))).astype(np.float32),
         "x_cond_bias": (0.1 * rng.standard_normal(L * 2 * R)).astype(np.float32),
         "x_geometry": np.array([Cc, T, window, stride, L, R, B])}
    want = host_cond(g, "x")                                     # nvwn_cond_from_features_host
    lib = _lib.lib()
    lib.nvwn_debug_get_conditioning.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int]
    n = T * stride

    def store(e):
        got = np.full((n, L, B, 2 * R), np.nan, np.float32)
        assert lib.nvwn_debug_get_conditioning(e._h, C.c_void_p(got.ctypes.data), first, n) == 0
        return got

    args = (g["x_features"], g["x_upsample_weight"], g["x_upsample_bias"], g["x_cond_weight"], g["x_cond_bias"], stride)
    e1 = nw.NVWavenetInfer(L, 2, B, N, R=R, S=256, A=256, dtype=nw.FP32)
    assert e1.set_conditioning_from_features(*args, first_sample=first) == n
    one_shot = store(e1)
    assert np.array_equal(one_shot.view(np.uint32), want.view(np.uint32)), np.abs(one_shot - want).max()

    e2 = nw.NVWavenetInfer(L, 2, B, N, R=R, S=256, A=256, dtype=nw.FP32)
    side = torch.cuda.Stream()
    assert e2.cond_producer_load(*args) == n
    for begin, count in ((0, 17), (17, 1), (18, n - 18)):
        e2.cond_producer_run(begin, count, first_sample=first, stream=side)
    side.synchronize()
    assert np.array_equal(store(e2).view(np.uint32), one_shot.view(np.uint32))
    with pytest.raises(Exception):
        e2.cond_producer_run(n - 2, 3, first_sample=first)       # past the loaded sequence
