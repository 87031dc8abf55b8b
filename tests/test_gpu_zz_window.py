"""Windowed engines (nvwn_create_windowed): every per-sample store holds W samples, sample t in slot t mod W, so one engine
generates utterances of any length in fixed device memory.

1. On each of the six kernel paths a windowed engine, fed chunk by chunk, gives the yOut of a full engine bit for bit, and the
   same last-step logits and probabilities; a run across the window edge is two launches.
2. NVWaveNet.generate (mel frames -> producer on a side stream -> windowed engine -> device mu-law) gives the audio of infer().
3. 720 utterances x 160 000 samples, more than a full engine could hold on the card, agree with a full engine on two tiles.
4. Sample indices near 2^31 give what the same inputs give at sample 0 (no 32-bit overflow of a sample-index product).
5. What a windowed engine refuses, with which code.
"""
import ctypes as C

import numpy as np
import pytest

import nv_wavenet_b200 as nw
from nv_wavenet_b200 import _lib
from tests import refgen
from tests.test_cond_producer import host_cond
from tests.test_gpu_parity import _select_fp16_kernel
from tests.test_window_abi import philox_at

pytestmark = pytest.mark.gpu

SEED = 0x77A1D0
LAT, TC, STREAM = nw.KERNEL_LATENCY, nw.KERNEL_TENSORCORE, nw.KERNEL_STREAM
EINVAL, EUNSUPPORTED = -1, -2                     # NVWN_EINVAL, NVWN_EUNSUPPORTED

# path -> (R, S, A, L, B, maxDil, dtype, fp16 kernel switch, expected kernel, expected cluster size); the fp16 paths have a
# 65-slot history ring, more than the 40-slot window: the window and the ring are independent
PATHS = {
    "lat_cluster": (64, 256, 256, 20, 8, 64, nw.FP16, "lat", LAT, 3),
    "lat_single": (64, 256, 256, 20, 8, 64, nw.FP16, "lat_single", LAT, 1),
    "tensorcore": (64, 256, 256, 20, 8, 64, nw.FP16, "tc", TC, 1),
    "fp16_stream": (128, 256, 256, 4, 3, 64, nw.FP16, None, STREAM, 1),       # R = 128: outside the mma kernels' shapes
    "fp32": (64, 256, 256, 8, 4, 8, nw.FP32, None, STREAM, 1),
    "fp32_fast": (64, 256, 256, 8, 4, 8, nw.FP32_FAST, None, STREAM, 1),
}
W, CHUNK, N = 40, 15, 97            # N > 2W and not a multiple of W; the chunk does not divide W


def _clear_env(monkeypatch):
    for k in ("NVWN_FP16_KERNEL", "NVWN_TC_TILE", "NVWN_TC_NODUP", "NVWN_TC_FUSED", "NVWN_LAT_CLUSTER", "NVWN_LAT_MAX_B"):
        monkeypatch.delenv(k, raising=False)


def run_range(e, init, count, num_samples, B, dump=False):
    """run_partial over samples [init, init + count) (the reference's run_partial + samples_per_chunk)."""
    e._samples_per_chunk = count
    try:
        e.run_partial(init, num_samples, B, None, 1, dump)
    finally:
        e._samples_per_chunk = 0


def windowed(L, md, B, window, R, S, A, dtype, w=None):
    e = nw.NVWavenetInfer(L, md, B, None, R=R, S=S, A=A, dtype=dtype, window=window)
    if w is not None:
        e.load(w)
    return e


@pytest.mark.parametrize("path", sorted(PATHS))
def test_windowed_equals_full_engine_bit_for_bit(path, monkeypatch):
    import torch
    R, S, A, L, B, md, dtype, switch, kernel, cluster = PATHS[path]
    _clear_env(monkeypatch)
    if switch:
        _select_fp16_kernel(switch, monkeypatch)
    w = refgen.lively_inputs(300 + R + L, R, S, A, L, B, N)

    full = nw.NVWavenetInfer(L, md, B, N, R=R, S=S, A=A, dtype=dtype)
    full.load(w)
    full.set_conditioning(w["Lh"], 0, N)
    full.set_selectors_random(SEED)
    full.reset_history()
    y_full = np.zeros((B, N), np.int32)
    full.run(N, B, y_full, dump_activations=True); full.synchronize()
    za_full, p_full = full.get_za(), full.get_p()
    assert (full.launch_info()["kernel"], full.launch_info()["cluster"]) == (kernel, cluster)
    assert len(np.unique(y_full)) > 8
    full.close()

    e = windowed(L, md, B, W, R, S, A, dtype, w)
    e.reset_history()
    y_win = np.full((B, N), -1, np.int32)
    for k, s0 in enumerate(range(0, N, CHUNK)):
        n = min(CHUNK, N - s0)
        lh = np.ascontiguousarray(w["Lh"][s0:s0 + n])
        src = lh if k % 2 == 0 else torch.from_numpy(lh).cuda()       # host and device sources in turn
        e.set_conditioning(src, s0, n)
        e.set_selectors_random_range(SEED, s0, n)
        before = e.launch_info()["launches"]
        run_range(e, s0, n, N, B, dump=s0 + n == N)
        crosses = s0 // W != (s0 + n - 1) // W
        assert e.launch_info()["launches"] - before == (2 if crosses else 1)
        part = np.zeros((B, n), np.int32)
        e.get_yout(part, s0, n)
        e.synchronize()
        y_win[:, s0:s0 + n] = part
        del src
    info = e.launch_info()
    assert (info["kernel"], info["cluster"]) == (kernel, cluster), info
    diff = np.nonzero((y_win != y_full).any(axis=0))[0]
    assert diff.size == 0, f"yOut differs from the full engine first at sample {diff[:1]}"
    assert np.array_equal(e.get_za().view(np.uint32), za_full.view(np.uint32))
    assert np.array_equal(e.get_p().view(np.uint32), p_full.view(np.uint32))
    # the last W samples in one read, across the window edge at 80
    last = np.zeros((B, W), np.int32)
    e.get_yout(last, N - W, W); e.synchronize()
    assert np.array_equal(last, y_full[:, N - W:])
    audio = e.get_audio(N - W, W, int16=True)
    lut = np.zeros(A, np.int16)
    assert _lib.lib().nvwn_mulaw_table(A, None, C.c_void_p(lut.ctypes.data), None) == 0
    assert np.array_equal(audio, lut[y_full[:, N - W:]])


def _net(w, L, md):
    """NVWaveNet over lively weights, as in test_gpu_parity.test_nvwavenet_python_class_matches_oracle."""
    import torch
    from nv_wavenet_b200.nv_wavenet import NVWaveNet
    R, S, A = 64, 256, 256
    tt = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    cm = lambda flat, M, K: np.ascontiguousarray(flat.reshape(K, M).T)
    return NVWaveNet(embedding_prev=tt(w["embPrev"]), embedding_curr=tt(w["embCur"]),
                     conv_out_weight=tt(cm(w["Wzs"], A, S)[:, :, None]), conv_end_weight=tt(cm(w["Wza"], A, A)[:, :, None]),
                     dilate_weights=[tt(np.stack([cm(w["Wprev"][l], 2 * R, R), cm(w["Wcur"][l], 2 * R, R)], axis=2)) for l in range(L)],
                     dilate_biases=[tt(w["Bh"][l]) for l in range(L)], max_dilation=md,
                     res_weights=[tt(cm(w["Wres"][l], R, R)[:, :, None]) for l in range(L - 1)],
                     res_biases=[tt(w["Bres"][l]) for l in range(L - 1)],
                     skip_weights=[tt(cm(w["Wskip"][l], S, R)[:, :, None]) for l in range(L)],
                     skip_biases=[tt(w["Bskip"][l]) for l in range(L)], use_embed_tanh=True)


def _mel(rng, B, Cc, T, window, L, R, lh_scale):
    return {"x_features": rng.standard_normal((B, Cc, T)).astype(np.float32),
            "x_upsample_weight": (0.3 / np.sqrt(Cc) * rng.standard_normal((Cc, Cc, window))).astype(np.float32),
            "x_upsample_bias": (0.1 * rng.standard_normal(Cc)).astype(np.float32),
            "x_cond_weight": (lh_scale / np.sqrt(Cc) * rng.standard_normal((L * 2 * R, Cc))).astype(np.float32),
            "x_cond_bias": (0.1 * lh_scale * rng.standard_normal(L * 2 * R)).astype(np.float32)}


def test_generate_streams_the_audio_of_infer(monkeypatch):
    import torch
    _clear_env(monkeypatch)
    R, L, md, B = 64, 12, 64, 8
    Cc, window, stride, chunk = 20, 16, 8, 64
    T = 28                                                       # 224 samples = 3.5 chunks
    rng = np.random.default_rng(17)
    w = refgen.lively_inputs(41, R, 256, 256, L, 1, 1)
    g = _mel(rng, B, Cc, T, window, L, R, 0.5)
    g["x_geometry"] = np.array([Cc, T, window, stride, L, R, B])
    net = _net(w, L, md)
    lh = host_cond(g, "x")                                       # nvwn_cond_from_features_host: [N][L][B][2R]
    n_total = T * stride
    cond = torch.from_numpy(np.ascontiguousarray(lh.transpose(3, 2, 1, 0))).cuda()
    net.infer(cond, 0, seed=SEED, fp16=True)
    want = net._engine(B, n_total, True).get_audio(0, n_total, int16=True)
    dev = lambda k: torch.from_numpy(g[k]).cuda()
    pieces = list(net.generate(dev("x_features"), dev("x_upsample_weight"), dev("x_upsample_bias"), dev("x_cond_weight"),
                               dev("x_cond_bias"), stride, chunk=chunk, seed=SEED, fp16=True))
    assert [(s0, a.shape[1]) for s0, a in pieces] == [(0, 64), (64, 64), (128, 64), (192, 32)]
    got = torch.cat([a for _, a in pieces], dim=1).cpu().numpy()
    assert got.dtype == np.int16 and len(np.unique(got)) > 16
    assert np.array_equal(got, want)
    eng = net._engines[(B, None, True, 2 * chunk)]
    assert eng.launch_info()["kernel"] == LAT and eng.launch_info()["cluster"] == 3


def test_long_form_beyond_device_memory(monkeypatch):
    """720 utterances x 160 000 samples (10 s at 16 kHz) at the C3 model on the three-CTA cluster kernel.  A full engine keeps
    L x 256 bytes of conditioning plus 12 bytes of selector, forcing and output per utterance-sample: 5 132 x 720 x 160 000 =
    591 GB, more than the card has; the windowed engine holds two 4 000-sample chunks (30 GB)."""
    import torch
    _clear_env(monkeypatch)
    R, S, A, L, md = 64, 256, 256, 20, 512
    B, n_total, chunk = 720, 160000, 4000
    Cc, window, stride = 80, 800, 200
    full_bytes = (L * 256 + 12) * B * n_total
    assert full_bytes > 590e9 and full_bytes > torch.cuda.get_device_properties(0).total_memory
    rng = np.random.default_rng(23)
    w = refgen.lively_inputs(43, R, S, A, L, 1, 1)
    g = _mel(rng, B, Cc, n_total // stride, window, L, R, 0.5)
    net = _net(w, L, md)
    dev = {k: torch.from_numpy(v).cuda() for k, v in g.items()}
    tiles = [0, B // 16 - 1]
    idx = np.array([b for t in tiles for b in range(16 * t, 16 * t + 16)])
    got = torch.empty((len(idx), n_total), dtype=torch.int16, device="cuda")
    gidx = torch.from_numpy(idx).cuda()
    for s0, audio in net.generate(dev["x_features"], dev["x_upsample_weight"], dev["x_upsample_bias"], dev["x_cond_weight"],
                                  dev["x_cond_bias"], stride, chunk=chunk, seed=SEED, fp16=True):
        got[:, s0:s0 + audio.shape[1]] = audio.index_select(0, gidx)
    eng = net._engines[(B, None, True, 2 * chunk)]
    assert (eng.launch_info()["kernel"], eng.launch_info()["cluster"]) == (LAT, 3)
    eng.close()
    net._engines.clear()
    torch.cuda.empty_cache()
    # a full engine holding only those 32 utterances (26 GB), with their selectors given explicitly
    small = net._engine(len(idx), n_total, True)
    small.set_conditioning_from_features(dev["x_features"].index_select(0, gidx).contiguous(), dev["x_upsample_weight"],
                                         dev["x_upsample_bias"], dev["x_cond_weight"], dev["x_cond_bias"], stride)
    t = np.arange(n_total, dtype=np.uint64)[:, None]
    small.set_selectors(philox_at(t * np.uint64(B) + idx.astype(np.uint64)[None, :], SEED))
    small.reset_history()
    small.run(n_total, len(idx), None)
    want = small.get_audio(0, n_total, int16=True)
    assert small.launch_info()["kernel"] == LAT
    got = got.cpu().numpy()
    diff = np.nonzero((got != want).any(axis=0))[0]
    assert diff.size == 0, f"audio differs from the full engine first at sample {diff[:1]}"
    assert len(np.unique(got)) > 64


@pytest.mark.parametrize("switch,kernel", [("lat", LAT), ("tc", TC), ("stream", STREAM)])
def test_high_sample_indices(switch, kernel, monkeypatch):
    """The same inputs placed at sample 0 and at 2^31 - n - 1 of two fresh engines give the same yOut: unwritten ring slots are
    zero, exactly like the t < d mask at the start of an utterance.  The high run crosses the window edge (two launches)."""
    R, S, A, L, B, md, n, win = 64, 256, 256, 20, 8, 8, 40, 48
    _clear_env(monkeypatch)
    _select_fp16_kernel(switch, monkeypatch)
    w = refgen.lively_inputs(61, R, S, A, L, B, n)
    ys = []
    for t0 in (0, 2 ** 31 - n - 1):
        e = windowed(L, md, B, win, R, S, A, nw.FP16, w)
        e.set_conditioning(w["Lh"], t0, n)
        e.set_selectors_range(w["selectors"], t0, n)
        run_range(e, t0, n, t0 + n, B)
        y = np.zeros((B, n), np.int32)
        e.get_yout(y, t0, n); e.synchronize()
        assert e.launch_info()["kernel"] == kernel
        assert e.launch_info()["launches"] == (1 if t0 == 0 else 2)
        ys.append(y)
        e.close()
    assert len(np.unique(ys[0])) > 8
    assert np.array_equal(ys[0], ys[1])


def test_windowed_contract(monkeypatch):
    _clear_env(monkeypatch)
    R, S, A, L, B, md, win = 64, 256, 256, 4, 2, 4, 16
    lib = _lib.lib()
    w = refgen.lively_inputs(5, R, S, A, L, B, 40)
    e = windowed(L, md, B, win, R, S, A, nw.FP32, w)
    h = e._h

    def err(rc, code, text):
        assert rc == code, (rc, lib.nvwn_last_error())
        assert text in lib.nvwn_last_error().decode()

    err(lib.nvwn_run_partial(h, 0, win + 1, 100, B, None, 0, None), EINVAL, "exceeds the window of 16")
    y = np.zeros((B, 40), np.int32)
    err(lib.nvwn_run_partial(h, 0, 4, 100, B, C.c_void_p(y.ctypes.data), 0, None), EINVAL, "yOut must be NULL")
    lh = np.zeros((win + 1, L, B, 2 * R), np.float32)
    err(lib.nvwn_set_conditioning(h, C.c_void_p(lh.ctypes.data), 3, win + 1, None), EINVAL, "17 samples exceed the window of 16")
    err(lib.nvwn_set_selectors_range(h, C.c_void_p(lh.ctypes.data), 0, win + 1, None), EINVAL, "exceed the window")
    err(lib.nvwn_set_conditioning(h, C.c_void_p(lh.ctypes.data), 2 ** 31 - 4, 4, None), EINVAL, "end at 2^31 - 1")
    sel = np.zeros((40, B), np.float32)
    err(lib.nvwn_set_inputs(h, C.c_void_p(lh.ctypes.data), C.c_void_p(sel.ctypes.data)), EUNSUPPORTED, "windowed engine")
    err(lib.nvwn_set_selectors(h, C.c_void_p(sel.ctypes.data)), EUNSUPPORTED, "windowed engine")
    err(lib.nvwn_set_selectors_random(h, C.c_ulonglong(1), None), EUNSUPPORTED, "windowed engine")
    err(lib.nvwn_set_forced(h, C.c_void_p(y.ctypes.data)), EUNSUPPORTED, "windowed engine")
    # outputs: only the last W samples generated since reset_history
    err(lib.nvwn_get_yout(h, C.c_void_p(y.ctypes.data), 0, 1, None), EINVAL, "not within the last window")
    e.reset_history()
    for s0 in range(0, 40, 10):
        e.set_conditioning(w["Lh"][s0:s0 + 10], s0, 10)
        e.set_selectors_random_range(SEED, s0, 10)
        run_range(e, s0, 10, 40, B)
    e.synchronize()
    assert lib.nvwn_get_yout(h, C.c_void_p(y.ctypes.data), 24, 16, None) == 0
    err(lib.nvwn_get_yout(h, C.c_void_p(y.ctypes.data), 23, 16, None), EINVAL, "not within the last window of generated samples [24, 40)")
    err(lib.nvwn_get_yout(h, C.c_void_p(y.ctypes.data), 30, 11, None), EINVAL, "not within the last window")
    a = np.zeros((B, 40), np.int16)
    err(lib.nvwn_get_audio(h, None, C.c_void_p(a.ctypes.data), 20, 4, 0, None), EINVAL, "not within the last window")
    assert lib.nvwn_get_audio(h, None, C.c_void_p(a.ctypes.data), 24, 4, 0, None) == 0
    e.reset_history()
    err(lib.nvwn_get_audio(h, None, C.c_void_p(a.ctypes.data), 24, 4, 0, None), EINVAL, "not within the last window")
    with pytest.raises(ValueError):
        nw.NVWavenetInfer(L, md, B, 40, R=R, S=S, A=A, window=win)
