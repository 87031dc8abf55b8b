"""SURVEY.md 8f next-1: persistent engine behind NVWaveNet.infer, device-side counter-based selectors, fp16 through the C-ABI."""
import ctypes as C

import numpy as np
import pytest

from tests import refgen
from tests.common import philox_selectors

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("dtype_name", ["fp32", "fp16"])
def test_device_selectors_equal_host_restatement(dtype_name):
    import nv_wavenet_b200 as nw
    R, S, A, L, B, N, md = 64, 256, 256, 5, 19, 40, 8
    w = refgen.lively_inputs(2, R, S, A, L, B, N)
    sel = philox_selectors(N * B, 0x1234ABCD5678).reshape(N, B)
    assert 0.0 <= sel.min() and sel.max() < 1.0 and abs(sel.mean() - 0.5) < 0.05
    dt = nw.FP16 if dtype_name == "fp16" else nw.FP32
    ys = []
    for mode in ("host", "device"):
        e = nw.NVWavenetInfer(L, md, B, N, R=R, S=S, A=A, dtype=dt)
        e.load(w); e.set_inputs(w["Lh"], sel)
        if mode == "device":
            e.set_selectors_random(0x1234ABCD5678)
        y = np.zeros((B, N), np.int32); e.run(N, B, y); e.synchronize()
        ys.append(y)
    assert np.array_equal(ys[0], ys[1]) and len(np.unique(ys[0])) > 16


def _net(w, L, R, S, A, md):
    import torch
    from nv_wavenet_b200.nv_wavenet import NVWaveNet
    tt = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to("cuda")
    cm = lambda flat, M, K: np.ascontiguousarray(flat.reshape(K, M).T)
    dilate = [tt(np.stack([cm(w["Wprev"][l], 2 * R, R), cm(w["Wcur"][l], 2 * R, R)], axis=2)) for l in range(L)]
    return NVWaveNet(embedding_prev=tt(w["embPrev"]), embedding_curr=tt(w["embCur"]),
                     conv_out_weight=tt(cm(w["Wzs"], A, S)[:, :, None]), conv_end_weight=tt(cm(w["Wza"], A, A)[:, :, None]),
                     dilate_weights=dilate, dilate_biases=[tt(w["Bh"][l]) for l in range(L)], max_dilation=md,
                     res_weights=[tt(cm(w["Wres"][l], R, R)[:, :, None]) for l in range(L - 1)],
                     res_biases=[tt(w["Bres"][l]) for l in range(L - 1)],
                     skip_weights=[tt(cm(w["Wskip"][l], S, R)[:, :, None]) for l in range(L)],
                     skip_biases=[tt(w["Bskip"][l]) for l in range(L)], use_embed_tanh=True)


def test_nvwavenet_keeps_one_engine_and_seeds_selectors():
    import torch
    from nv_wavenet_b200.nv_wavenet import Impl
    R, S, A, L, B, N, md = 64, 256, 256, 4, 3, 24, 4
    w = refgen.lively_inputs(7, R, S, A, L, B, N)
    net = _net(w, L, R, S, A, md)
    cond = torch.from_numpy(np.ascontiguousarray(w["Lh"].transpose(3, 2, 1, 0))).cuda()
    y1 = net.infer(cond, Impl.AUTO, seed=11).cpu().numpy()
    y2 = net.infer(cond, Impl.PERSISTENT, seed=11).cpu().numpy()
    y3 = net.infer(cond, Impl.AUTO, seed=12).cpu().numpy()
    assert net.engines_created == 1, "weights must be uploaded once, not per call"
    assert np.array_equal(y1, y2) and not np.array_equal(y1, y3)
    # libc mode (seed=None) replays with srand, like the reference wrapper
    libc = C.CDLL(None)
    libc.srand(5); ya = net.infer(cond, Impl.AUTO).cpu().numpy()
    libc.srand(5); yb = net.infer(cond, Impl.AUTO).cpu().numpy()
    assert np.array_equal(ya, yb) and net.engines_created == 1
    # fp16 engine is a second persistent engine of the same object
    yh = net.infer(cond, Impl.AUTO, seed=11, fp16=True).cpu().numpy()
    assert net.engines_created == 2 and yh.shape == y1.shape and (yh == y1).mean() > 0.3


def test_wavenet_infer_fp16_entry_point():
    """The fp16 C-ABI entry (same arguments as wavenet_infer): equals the engine's fp16 run on the same libc selectors."""
    import nv_wavenet_b200 as nw
    from nv_wavenet_b200 import _lib
    lib = _lib.lib()
    R, S, A = lib.get_R(), lib.get_S(), lib.get_A()
    L, B, N, md = 4, 5, 20, 4
    w = refgen.lively_inputs(78, R, S, A, L, B, N)
    libc = C.CDLL(None)
    libc.srand(4321)
    arr = lambda key: (C.c_void_p * L)(*[w[key][l].ctypes.data for l in range(L)])
    samples = np.zeros((B, N), np.int32)
    lib.wavenet_infer_fp16(N, B, w["embPrev"].ctypes.data, w["embCur"].ctypes.data, L, md,
                           arr("Wprev"), arr("Wcur"), arr("Bh"), arr("Wres"), arr("Bres"), arr("Wskip"), arr("Bskip"),
                           w["Wzs"].ctypes.data, w["Wza"].ctypes.data, 1, w["Lh"].ctypes.data, 0, samples.ctypes.data)
    rng = refgen.GlibcRand(4321)
    sel = refgen.randomize(rng, B, N, np.float32(0.5), np.float32(1.0)).reshape(N, B)
    w2 = dict(w); w2["Bzs"] = np.zeros(A, np.float32); w2["Bza"] = np.zeros(A, np.float32)
    e = nw.NVWavenetInfer(L, md, B, N, R=R, S=S, A=A, dtype=nw.FP16)
    e.load(w2); e.set_inputs(w["Lh"], sel)
    y = np.zeros((B, N), np.int32); e.run(N, B, y); e.synchronize()
    assert np.array_equal(samples, y) and len(np.unique(y)) > 8
