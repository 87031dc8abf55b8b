"""Generates tests/golden/cond_input.npz with the reference's own conditioning path (pytorch/wavenet.py:57-70,190-202:
WaveNet.upsample, WaveNet.cond_layers, WaveNet.get_cond_input) on the CPU in the build container, and the permute
pytorch/nv_wavenet.py applies before calling the kernel ([2R][B][L][N] -> [N][L][B][2R]).
/root/reference does not exist on the GPU box: only the committed .npz travels.

    python tests/golden/make_golden_cond.py

<name>_Lh holds every <name>_Lh_stride-th element of the flattened [N][L][B][2R] tensor, which keeps the file under 1 MB.
A stride coprime with 2R, B and L samples every channel, utterance and layer.
"""
import os
import sys
import warnings

import numpy as np
import torch

sys.path.insert(0, "/root/reference/pytorch")
warnings.simplefilter("ignore")
import wavenet as ref_wavenet  # noqa: E402  (the reference's module)

out = {}
#        name   C   T  window stride  L   R   B  Lh stride
cases = [("a", 8, 2, 800, 200, 2, 32, 2, 1),      # the reference's upsampling geometry (config.json: window 800, stride 200), 8 bands to keep the file small
         ("b", 5, 7, 12, 4, 3, 4, 3, 1),          # odd small geometry: window = 3 strides
         ("c", 6, 3, 40, 10, 4, 64, 19, 5)]       # R = 64 (the tensor-core / latency kernels' tiled fp16 layouts), two 16-utterance tiles, ragged
for name, C, T, window, stride, L, R, B, lh_stride in cases:
    torch.manual_seed(1234 + C)
    m = ref_wavenet.WaveNet(n_in_channels=256, n_layers=L, max_dilation=2, n_residual_channels=R, n_skip_channels=16,
                            n_out_channels=256, n_cond_channels=C, upsamp_window=window, upsamp_stride=stride)
    feats = torch.randn(B, C, T)
    with torch.no_grad():
        cond = m.get_cond_input(feats)                                  # [2R][B][L][N]
        lh = cond.permute(3, 2, 1, 0).contiguous()                      # [N][L][B][2R], what the kernel consumes
    out.update({f"{name}_features": feats.numpy(), f"{name}_upsample_weight": m.upsample.weight.detach().numpy(),
                f"{name}_upsample_bias": m.upsample.bias.detach().numpy(),
                f"{name}_cond_weight": m.cond_layers.conv.weight.detach().numpy()[:, :, 0],
                f"{name}_cond_bias": m.cond_layers.conv.bias.detach().numpy(), f"{name}_Lh": lh.numpy().reshape(-1)[::lh_stride],
                f"{name}_Lh_stride": np.array(lh_stride), f"{name}_geometry": np.array([C, T, window, stride, L, R, B])})
    print(name, tuple(lh.shape), float(lh.abs().max()))
np.savez_compressed(os.path.join(os.path.dirname(__file__), "cond_input.npz"), **out)
