"""PyTorch-facing binding with the surface of the reference's `pytorch/nv_wavenet.py` -- class `NVWaveNet`, the `Impl`
constants and `column_major` -- implemented over the handle C-ABI (include/nvwn_b200.h) through ctypes (the reference's
THC-era pybind wrapper, `pytorch/wavenet_infer_wrapper.cpp`, no longer builds against torch >= 2).

    wavenet = NVWaveNet(**model.export_weights())
    samples = wavenet.infer(cond_input, Impl.PERSISTENT)      # int32 CUDA tensor [batch, samples]

Unlike the reference wrapper (pytorch/wavenet_infer.cu:87-145 builds the whole nvWavenetInfer object, uploads every weight and
frees it again on EVERY call) the object keeps a persistent engine per (batch, samples, precision): weights are uploaded once,
infer() only sets the inputs.  Selectors: `seed=None` draws them like the reference (libc rand(), replayable with srand());
an integer seed draws them on the device (counter-based Philox, include/nvwn_b200.h).

`generate()` streams audio of any length from mel frames: a windowed engine (fixed device memory whatever the length), the
conditioning produced on the device one chunk ahead on a side stream, and the mu-law decode on the device.

Constructor arguments, accepted shapes, the appended unused residual layer and the memory layouts handed to the
kernel are those of pytorch/nv_wavenet.py:55-196; the code is organised around one table of expected shapes.
"""
import ctypes as C

import torch

from . import _lib


class Impl:
    """`implementation` argument of infer() (pytorch/nv_wavenet.py:51-54); one kernel family serves all of them here."""
    AUTO = 0
    SINGLE_BLOCK = 1
    DUAL_BLOCK = 2
    PERSISTENT = 3


def column_major(x):
    """Row-major torch tensor -> the column-major layout the kernel reads (pytorch/nv_wavenet.py:33-49):
    vectors unchanged, [M][K] and conv-style [M][K][1] matrices transposed, 4-D conditioning fully reversed."""
    nd = x.dim()
    if nd == 1:
        return x
    if nd == 3:
        if x.size(2) != 1:
            raise AssertionError("column_major: 3-D tensors must be convolution weights of kernel size 1")
        x, nd = x[:, :, 0], 2
    if nd == 2:
        return x.t().contiguous()
    if nd == 4:
        return x.permute(3, 2, 1, 0).contiguous()
    raise AssertionError(f"column_major: unsupported rank {nd}")


def _expect(name, tensor, shape):
    got = tuple(tensor.size())[:len(shape)]
    if got != tuple(shape):
        raise AssertionError(f"{name}: shape {got} does not match the compiled kernel's {tuple(shape)}")


class NVWaveNet:
    def __init__(self, embedding_prev, embedding_curr, conv_out_weight, conv_end_weight, dilate_weights, dilate_biases,
                 max_dilation, res_weights, res_biases, skip_weights, skip_biases, use_embed_tanh):
        self._lib = _lib.lib()
        R, S, A = self._lib.get_R(), self._lib.get_S(), self._lib.get_A()
        self.R, self.S, self.A = R, S, A
        self.max_dilation = max_dilation
        self.use_embed_tanh = use_embed_tanh

        # embeddings arrive [A][R] and are consumed as emb[a * R + r]: two transposes cancel, keep the values as they are
        _expect("embedding_prev", embedding_prev, (A, R))
        _expect("embedding_curr", embedding_curr, (A, R))
        self.embedding_prev = column_major(embedding_prev.t())
        self.embedding_curr = column_major(embedding_curr.t())
        _expect("conv_out_weight", conv_out_weight, (A, S))
        _expect("conv_end_weight", conv_end_weight, (A, A))
        self.conv_out = column_major(conv_out_weight)
        self.conv_end = column_major(conv_end_weight)

        n = len(dilate_weights)
        counts = {"dilate_biases": len(dilate_biases), "skip_weights": len(skip_weights), "skip_biases": len(skip_biases),
                  "res_weights": len(res_weights) + 1, "res_biases": len(res_biases) + 1}      # the last layer has no residual conv
        if any(c != n for c in counts.values()):
            raise AssertionError(f"Number of layers is inconsistent for different parameter types: dilate_weights {n}, {counts}")
        # the kernel still wants a residual matrix for the last layer: all zero (pytorch/nv_wavenet.py:139-141)
        like = dilate_weights[0] if n else embedding_prev
        res_weights = list(res_weights) + [torch.zeros(R, R, dtype=like.dtype, device=like.device)]
        res_biases = list(res_biases) + [torch.zeros(R, dtype=like.dtype, device=like.device)]

        self.layers = []                                 # per layer: (Wprev, Wcur, Bh, Wres, Bres, Wskip, Bskip), kernel layouts
        for l in range(n):
            w = dilate_weights[l]
            if w.size(2) != 2:
                raise AssertionError("nv-wavenet only supports kernel_size 2 dilated convolutions")
            _expect(f"dilate_weights[{l}]", w, (2 * R, R))
            _expect(f"dilate_biases[{l}]", dilate_biases[l], (2 * R,))
            _expect(f"res_weights[{l}]", res_weights[l], (R, R))
            _expect(f"res_biases[{l}]", res_biases[l], (R,))
            _expect(f"skip_weights[{l}]", skip_weights[l], (S, R))
            _expect(f"skip_biases[{l}]", skip_biases[l], (S,))
            self.layers.append((column_major(w[:, :, 0]), column_major(w[:, :, 1]), dilate_biases[l],
                                column_major(res_weights[l]), res_biases[l], column_major(skip_weights[l]), skip_biases[l]))
        self.num_layers = n
        self._engines = {}                               # (batch, samples, fp16, window) -> persistent NVWavenetInfer
        self.engines_created = 0

    def _engine(self, batch_size, sample_count, fp16, window=None):
        """The persistent engine for this problem size (created and loaded on first use); a windowed one if `window` is given."""
        from .infer import NVWavenetInfer
        key = (batch_size, sample_count, bool(fp16), window)
        eng = self._engines.get(key)
        if eng is None:
            eng = NVWavenetInfer(self.num_layers, self.max_dilation, batch_size, sample_count, 0, bool(self.use_embed_tanh),
                                 R=self.R, S=self.S, A=self.A, dtype=_lib.FP16 if fp16 else _lib.FP32, window=window)
            f32 = lambda t: t.float().contiguous()
            eng.set_embeddings(f32(self.embedding_prev), f32(self.embedding_curr))
            for l, layer in enumerate(self.layers):
                eng.set_layer_weights(l, *[f32(t) for t in layer])
            zero = torch.zeros(self.A, dtype=torch.float32)                 # "We didn't use biases on our outputs" (wavenet_infer.cu:75-82)
            eng.set_out_weights(f32(self.conv_out), zero, f32(self.conv_end), zero)
            self._engines[key] = eng
            self.engines_created += 1
        return eng

    def infer(self, cond_input, implementation, seed=None, fp16=False):
        """cond_input: channels x batch x num_layers x samples (pytorch/nv_wavenet.py:172-196); returns int32 [batch][samples].
        `implementation` (Impl.*) is accepted for compatibility: one kernel family serves all of them."""
        if (cond_input.size(0), cond_input.size(2)) != (2 * self.R, self.num_layers):
            raise AssertionError(f"Inputs are channels x batch x num_layers x samples; got {tuple(cond_input.size())}")
        batch_size, sample_count = cond_input.size(1), cond_input.size(3)
        eng = self._engine(batch_size, sample_count, fp16)
        lh = column_major(cond_input).float()                       # [samples][layers][batch][2R]
        eng.reset_history()
        eng.set_conditioning(lh, 0, sample_count)
        if seed is None:                                            # the reference's host draw, on the caller's rand() stream
            import numpy as np
            sel = np.empty(sample_count * batch_size, np.float32)
            _lib.check(self._lib.nvwn_libc_selectors(C.c_void_p(sel.ctypes.data), batch_size, sample_count), "selectors")
            eng.set_selectors(sel)
        else:
            eng.set_selectors_random(seed)
        samples = torch.empty((batch_size, sample_count), dtype=torch.int32, device="cuda")
        eng.run(sample_count, batch_size, samples, dump_activations=False)
        torch.cuda.synchronize()
        return samples

    def generate(self, features, upsample_weight, upsample_bias, cond_weight, cond_bias, stride, chunk=8000, seed=0, fp16=False):
        """Streams the audio of mel frames `features` [B][C][T] chunk by chunk: yields (first_sample, audio) with `audio` an int16
        CUDA tensor [B][n] (the reference's post-processing, saturate off), ordered on the current stream.

        The upsampling and cond layers are those of set_conditioning_from_features (upsample_weight [C][C][window], cond_weight
        [L*2R][C]).  One persistent windowed engine per (batch, chunk, precision) with a window of two chunks holds the utterance,
        so device memory does not grow with T.  Chunk k+1's conditioning is produced on a side stream while chunk k generates;
        it overwrites the slots of chunk k-1 only after that chunk's audio is decoded.  Selectors are the counter-based ones of
        `seed`, so the audio equals infer(cond_input, seed=seed) on the same conditioning."""
        B = features.size(0)
        eng = self._engine(B, None, fp16, window=2 * chunk)
        total = eng.cond_producer_load(features, upsample_weight, upsample_bias, cond_weight, cond_bias, stride)
        eng.reset_history()
        main, side = torch.cuda.current_stream(), torch.cuda.Stream()
        starts = list(range(0, total, chunk))
        produced, decoded = [], []

        def produce(k):
            s0 = starts[k]
            if k == 0:
                side.wait_stream(main)                                  # any earlier use of the engine on this stream
            if k >= 2:
                side.wait_event(decoded[k - 2])                         # chunk k takes the slots of chunk k - 2
            eng.cond_producer_run(s0, min(chunk, total - s0), stream=side)
            ev = torch.cuda.Event()
            ev.record(side)
            produced.append(ev)

        produce(0)
        for k, s0 in enumerate(starts):
            n = min(chunk, total - s0)
            if k + 1 < len(starts):
                produce(k + 1)
            eng.set_selectors_random_range(seed, s0, n, stream=main)
            main.wait_event(produced[k])
            eng._samples_per_chunk = n
            try:
                eng.run_partial(s0, total, B, None, 1, False, main)
            finally:
                eng._samples_per_chunk = 0
            audio = torch.empty((B, n), dtype=torch.int16, device="cuda")
            eng.get_audio(s0, n, int16=True, out=audio, stream=main)
            ev = torch.cuda.Event()
            ev.record(main)
            decoded.append(ev)
            yield s0, audio
