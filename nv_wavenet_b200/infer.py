"""Host-side mirror of the reference's C++ class nvWavenetInfer<T_weight,T_data,R,S,A>
(nv_wavenet.cuh:220-640) over the C-ABI in include/nvwn_b200.h.

Same member names and argument meaning as the reference class; array arguments may be numpy
arrays (host memory) or CUDA torch tensors (device memory) -- the reference setters also accept
either kind of pointer (nv_wavenet.cuh:285-308).  All compute happens in the CUDA library.
"""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import FP16, FP32, FP32_FAST, KERNEL_AUTO, KERNEL_STREAM, KERNEL_TENSORCORE, check  # noqa: F401

# Implementation enum of the reference (nv_wavenet.cuh:223-229); accepted, all map to the sm_100a kernels
AUTO, SINGLE_BLOCK, DUAL_BLOCK, PERSISTENT, MANYBLOCK_NONPERSISTENT = 0, 1, 2, 3, 4


def _ptr(a, dtype):
    """(void*, keepalive) of a numpy array or torch tensor holding `dtype`, C-contiguous."""
    if a is None:
        return None, None
    if isinstance(a, np.ndarray):
        if a.dtype != dtype or not a.flags["C_CONTIGUOUS"]:
            a = np.ascontiguousarray(a, dtype=dtype)
        return C.c_void_p(a.ctypes.data), a
    if hasattr(a, "data_ptr"):          # torch tensor (host or device)
        import torch
        want = torch.float32 if dtype == np.float32 else torch.int32
        if a.dtype != want or not a.is_contiguous():
            a = a.to(want).contiguous()
        return C.c_void_p(a.data_ptr()), a
    a = np.ascontiguousarray(a, dtype=dtype)
    return C.c_void_p(a.ctypes.data), a


def _stream(stream):
    if stream is None:
        return None
    if hasattr(stream, "cuda_stream"):
        return C.c_void_p(stream.cuda_stream)
    return C.c_void_p(int(stream))


class NVWavenetInfer:
    """nvWavenetInfer(numLayers, maxDilation, batchSize, numSamples, impl=0, tanhEmbed=True)
    with the template parameters (precision, R, S, A) as keyword arguments.

    `window=W` with `num_samples=None` creates a windowed engine (nvwn_create_windowed): its stores hold W samples, sample t in
    slot t % W, so it generates utterances of any length in fixed device memory.  Sample ranges are absolute; see
    include/nvwn_b200.h for what a windowed engine accepts."""

    def __init__(self, num_layers, max_dilation, batch_size, num_samples, impl=AUTO, tanh_embed=True,
                 *, R=64, S=128, A=256, dtype=FP32, window=None):
        self._l = _lib.lib()
        if (num_samples is None) == (window is None):
            raise ValueError("give num_samples (a full engine) or window (a windowed engine), not both")
        self.L, self.max_dilation, self.B, self.N, self.W = num_layers, max_dilation, batch_size, num_samples, window
        self.R, self.S, self.A, self.dtype = R, S, A, dtype
        h = C.c_void_p()
        create = self._l.nvwn_create if window is None else self._l.nvwn_create_windowed
        check(create(C.byref(h), dtype, R, S, A, num_layers, max_dilation, batch_size, num_samples if window is None else window,
                     impl, int(bool(tanh_embed))), "nvwn_create" if window is None else "nvwn_create_windowed")
        self._h = h
        self._samples_per_chunk = 0

    def close(self):
        if getattr(self, "_h", None):
            self._l.nvwn_destroy(self._h)
            self._h = None

    __del__ = close

    # ---- model initialisation (nv_wavenet.cuh:396-415) ----
    def set_embeddings(self, embed_prev, embed_cur):
        p, k1 = _ptr(embed_prev, np.float32); c, k2 = _ptr(embed_cur, np.float32)
        check(self._l.nvwn_set_embeddings(self._h, p, c), "setEmbeddings")

    def set_layer_weights(self, layer, Wprev, Wcur, Bh, Wres, Bres, Wskip, Bskip):
        ptrs = [_ptr(a, np.float32) for a in (Wprev, Wcur, Bh, Wres, Bres, Wskip, Bskip)]
        check(self._l.nvwn_set_layer_weights(self._h, layer, *[p for p, _ in ptrs]), "setLayerWeights")

    def set_out_weights(self, Wzs, Bzs, Wza, Bza):
        ptrs = [_ptr(a, np.float32) for a in (Wzs, Bzs, Wza, Bza)]
        check(self._l.nvwn_set_out_weights(self._h, *[p for p, _ in ptrs]), "setOutWeights")

    def load(self, w):
        """Convenience: dict with embPrev, embCur, Wprev[L], ... as produced by tests/refgen.py."""
        self.set_embeddings(w["embPrev"], w["embCur"])
        for l in range(self.L):
            self.set_layer_weights(l, w["Wprev"][l], w["Wcur"][l], w["Bh"][l], w["Wres"][l], w["Bres"][l],
                                   w["Wskip"][l], w["Bskip"][l])
        self.set_out_weights(w["Wzs"], w["Bzs"], w["Wza"], w["Bza"])

    # ---- inputs (nv_wavenet.cuh:417-422) ----
    def set_inputs(self, Lh, output_selectors):
        a, k1 = _ptr(Lh, np.float32); s, k2 = _ptr(output_selectors, np.float32)
        check(self._l.nvwn_set_inputs(self._h, a, s), "setInputs")

    def set_selectors(self, output_selectors):
        s, k = _ptr(output_selectors, np.float32)
        check(self._l.nvwn_set_selectors(self._h, s), "setSelectors")

    def set_selectors_random(self, seed, stream=None):
        """Selectors drawn on the device: counter-based (Philox-4x32-10, key = seed), see include/nvwn_b200.h."""
        check(self._l.nvwn_set_selectors_random(self._h, C.c_ulonglong(int(seed) & (2 ** 64 - 1)), _stream(stream)), "setSelectorsRandom")

    def set_selectors_range(self, selectors, first_sample, num_samples, stream=None):
        """Selectors of samples [first_sample, first_sample + num_samples) only: float32 [num_samples][B], host or device."""
        s, k = _ptr(selectors, np.float32)
        check(self._l.nvwn_set_selectors_range(self._h, s, first_sample, num_samples, _stream(stream)), "setSelectorsRange")
        return k

    def set_selectors_random_range(self, seed, first_sample, num_samples, stream=None):
        """The values set_selectors_random(seed) gives samples [first_sample, first_sample + num_samples), drawn for those only."""
        check(self._l.nvwn_set_selectors_random_range(self._h, C.c_ulonglong(int(seed) & (2 ** 64 - 1)), first_sample, num_samples,
                                                      _stream(stream)), "setSelectorsRandomRange")

    def set_conditioning(self, Lh, first_sample, num_samples, stream=None):
        a, k = _ptr(Lh, np.float32)
        check(self._l.nvwn_set_conditioning(self._h, a, first_sample, num_samples, _stream(stream)), "setConditioning")
        return k

    def set_conditioning_from_features(self, features, upsample_weight, upsample_bias, cond_weight, cond_bias, stride,
                                       first_sample=0, stream=None):
        """Device-side WaveNet.get_cond_input (pytorch/wavenet.py:190-202) + the permutes of pytorch/nv_wavenet.py:48-49,181:
        features [B][C][T], upsample_weight [C][C][window] (ConvTranspose1d), cond_weight [L*2R][C] (or [L*2R][C][1]),
        numpy arrays or torch tensors (host or CUDA).  Fills conditioning for T*stride samples from `first_sample`."""
        shp = lambda a: tuple(a.shape)
        B, Cc, T = shp(features)
        assert B == self.B and shp(upsample_weight)[:2] == (Cc, Cc) and shp(cond_weight)[:2] == (self.L * 2 * self.R, Cc)
        window = shp(upsample_weight)[2]
        f, k1 = _ptr(features, np.float32); wu, k2 = _ptr(upsample_weight, np.float32); bu, k3 = _ptr(upsample_bias, np.float32)
        wc, k4 = _ptr(cond_weight, np.float32); bc, k5 = _ptr(cond_bias, np.float32)
        check(self._l.nvwn_set_conditioning_from_features(self._h, f, Cc, T, wu, bu, window, stride, wc, bc, first_sample,
                                                          _stream(stream)), "setConditioningFromFeatures")
        return T * stride

    def cond_producer_load(self, features, upsample_weight, upsample_bias, cond_weight, cond_bias, stride, stream=None):
        """First half of set_conditioning_from_features: copies the features and both layers' weights into engine-owned device
        memory.  Returns the number of samples the sequence covers (T * stride)."""
        shp = lambda a: tuple(a.shape)
        B, Cc, T = shp(features)
        assert B == self.B and shp(upsample_weight)[:2] == (Cc, Cc) and shp(cond_weight)[:2] == (self.L * 2 * self.R, Cc)
        window = shp(upsample_weight)[2]
        f, k1 = _ptr(features, np.float32); wu, k2 = _ptr(upsample_weight, np.float32); bu, k3 = _ptr(upsample_bias, np.float32)
        wc, k4 = _ptr(cond_weight, np.float32); bc, k5 = _ptr(cond_bias, np.float32)
        check(self._l.nvwn_cond_producer_load(self._h, f, Cc, T, wu, bu, window, stride, wc, bc, _stream(stream)), "condProducerLoad")
        return T * stride

    def cond_producer_run(self, sample_begin, sample_count, first_sample=0, stream=None):
        """Second half: conditioning of samples [sample_begin, sample_begin + sample_count) of the loaded sequence, asynchronously on
        `stream` (record an event after it and make the generating stream wait for it)."""
        check(self._l.nvwn_cond_producer_run(self._h, first_sample, sample_begin, sample_count, _stream(stream)), "condProducerRun")

    def reset_history(self):
        check(self._l.nvwn_reset_history(self._h), "resetHistory")

    def set_forced(self, forced):
        f, k = _ptr(forced, np.int32)
        check(self._l.nvwn_set_forced(self._h, f), "setForced")

    # ---- fetch intermediate results (nv_wavenet.cuh:424-444) ----
    def _get(self, fn, shape, *pre):
        out = np.empty(shape, np.float32)
        check(getattr(self._l, fn)(self._h, *pre, C.c_void_p(out.ctypes.data)), fn)
        return out

    def get_xt_out(self, layer): return self._get("nvwn_get_xt_out", (self.B, self.R), layer)
    def get_skip_out(self, layer): return self._get("nvwn_get_skip_out", (self.B, self.S), layer)
    def get_zs(self): return self._get("nvwn_get_zs", (self.B, self.A))
    def get_za(self): return self._get("nvwn_get_za", (self.B, self.A))
    def get_p(self): return self._get("nvwn_get_p", (self.B, self.A))

    def activations(self):
        return {"xt": np.stack([self.get_xt_out(l) for l in range(self.L)]),
                "skip": np.stack([self.get_skip_out(l) for l in range(self.L)]),
                "zs": self.get_zs(), "za": self.get_za(), "p": self.get_p()}

    def get_yout(self, y_out, offset, size, stream=None):
        p, k = _ptr(y_out, np.int32)
        check(self._l.nvwn_get_yout(self._h, p, offset, size, _stream(stream)), "getYOut")

    def get_audio(self, offset=0, size=None, int16=False, saturate=False, out=None, stream=None):
        """Device-side replacement of the reference's host post-processing (pytorch/nv_wavenet_inference.py:55-60):
        mu-law decode (utils.mu_law_decode_numpy, mu_quantization = A) of yOut[:, offset:offset+size], as float32
        in [-1, 1] or, with int16=True, as `(MAX_WAV_VALUE * audio).astype('int16')`.  `out`: numpy array or torch
        tensor [B][size] of the matching dtype (a CUDA tensor is filled asynchronously on `stream`); allocated
        (numpy) if None.  saturate=False keeps the reference's cast of the top code (+1.0 -> -32768).  On a windowed engine
        `offset` is an absolute sample index and `size` must be given."""
        if size is None:
            if self.W is not None:
                raise ValueError("get_audio on a windowed engine needs `size`")
            size = self.N - offset
        if out is None:
            out = np.empty((self.B, size), np.int16 if int16 else np.float32)
        if isinstance(out, np.ndarray):
            assert out.flags["C_CONTIGUOUS"] and out.dtype == (np.int16 if int16 else np.float32) and out.size == self.B * size
            p = C.c_void_p(out.ctypes.data)
        else:                               # torch tensor
            import torch
            assert out.is_contiguous() and out.dtype == (torch.int16 if int16 else torch.float32) and out.numel() == self.B * size
            p = C.c_void_p(out.data_ptr())
        check(self._l.nvwn_get_audio(self._h, None if int16 else p, p if int16 else None, offset, size, int(saturate),
                                     _stream(stream)), "getAudio")
        return out

    # ---- run (nv_wavenet.cuh:445-639) ----
    def run_partial(self, init_sample, num_samples, batch_size, y_out=None, batch_size_per_block=1,
                    dump_activations=False, stream=None):
        count = self._samples_per_chunk if self._samples_per_chunk else num_samples
        p, k = _ptr(y_out, np.int32)
        check(self._l.nvwn_run_partial(self._h, init_sample, count, num_samples, batch_size, p,
                                       int(dump_activations), _stream(stream)), "run_partial")
        return True

    def run(self, num_samples, batch_size, y_out=None, batch_size_per_block=1, dump_activations=False, stream=None):
        """Returns True like the reference; y_out (numpy int32 [B][N] or CUDA int tensor) is filled
        asynchronously on `stream` exactly as the reference does -- synchronize() before reading."""
        self._samples_per_chunk = 0
        return self.run_partial(0, num_samples, batch_size, y_out, batch_size_per_block, dump_activations, stream)

    def run_chunks(self, num_samples_per_chunk, consume, num_samples, batch_size, y_out=None,
                   batch_size_per_block=1, dump_activations=False, stream=None):
        """run_chunks (nv_wavenet.cuh:445-497): launch chunk after chunk; each chunk of yOut is copied
        out on a second stream as soon as it is produced; consume(yOut, initSample, count) per chunk."""
        import torch
        compute = stream if stream is not None else torch.cuda.current_stream()
        copy = torch.cuda.Stream()
        chunks = []
        for init in range(0, num_samples, num_samples_per_chunk):
            n = min(num_samples_per_chunk, num_samples - init)
            self._samples_per_chunk = n
            self.run_partial(init, num_samples, batch_size, None, batch_size_per_block, True, compute)
            ev = torch.cuda.Event(); ev.record(compute)
            copy.wait_event(ev)
            if y_out is not None:
                self.get_yout(y_out, init, n, copy)
            done = torch.cuda.Event(); done.record(copy)
            chunks.append((init, n, done))
        self._samples_per_chunk = 0
        for init, n, done in chunks:
            done.synchronize()
            consume(y_out, init, n)
        return True

    def synchronize(self):
        import torch
        torch.cuda.synchronize()

    def launch_info(self):
        info = _lib.LaunchInfo()
        check(self._l.nvwn_get_launch_info(self._h, C.byref(info)), "launch_info")
        return {k: getattr(info, k) for k, _ in _lib.LaunchInfo._fields_}

    def weight_blob(self):
        p = C.c_void_p(); n = C.c_ulonglong()
        check(self._l.nvwn_weight_blob(self._h, C.byref(p), C.byref(n)), "weight_blob")
        return p.value, n.value

    def weights_updated(self):
        check(self._l.nvwn_weights_updated(self._h), "weights_updated")
