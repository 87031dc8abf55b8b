"""Generates tests/golden/reference_gpu.npz with the reference's OWN CUDA kernels (oracle/_ref/ref_gpu_harness, built by
`make -C oracle refgpu` where the reference sources are present) on a GPU, for tests/test_gpu_vs_reference_gpu.py:

    python tests/golden/make_golden_ref_gpu.py [output.npz]

For each case (fp32, fp16): <case>/in_sha (sha256 of the inputs, which the test regenerates), <case>/y int32 [B][N]
sampled indices and <case>/za float32 [B][A] logits of the last sample, from the PERSISTENT kernel (mode 3).
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import ref_gpu                          # noqa: E402
from tests import common                            # noqa: E402
from tests import test_gpu_vs_reference_gpu as t    # noqa: E402


def main():
    path = sys.argv[1] if len(sys.argv) > 1 else t.GOLDEN
    out = {}
    for name, case, precision, chunk in (("fp32", t.fp32_case, 32, 7), ("fp16", t.fp16_case, 16, 2048)):
        w, B, N = case()
        ref = ref_gpu.run(w, precision, t.R, t.S, t.A, t.L, t.MD, B, N, mode=3, chunk=chunk)
        out[name + "/in_sha"] = np.array(common.sha([w[k] for k in common.INPUT_KEYS]))
        out[name + "/y"] = ref["y"]
        out[name + "/za"] = ref["za"]
        print(name, "distinct indices", len(np.unique(ref["y"])), "max |za|", float(np.abs(ref["za"]).max()))
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
