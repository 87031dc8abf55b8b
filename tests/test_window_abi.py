"""CPU-side checks of the windowed-engine entry points: the header declares them and the library exports them, and the host
restatement of the counter-based selectors drawn for a range of samples (Philox counter sample * B + b) is the slice of the
whole draw."""
import os
import re

import numpy as np

from nv_wavenet_b200 import _lib
from tests.common import philox_selectors

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW = ("nvwn_create_windowed", "nvwn_set_selectors_range", "nvwn_set_selectors_random_range")


def philox_at(ctr, seed):
    """wn_philox_first (csrc/wn_convert.cu) at arbitrary 64-bit counters `ctr` (any shape), mapped to [0, 1) with 24 bits."""
    ctr = np.asarray(ctr, np.uint64)
    M = np.uint64(0xFFFFFFFF)
    c0, c1 = ctr & M, ctr >> np.uint64(32)
    c2 = np.zeros_like(ctr); c3 = np.zeros_like(ctr)
    k0, k1 = np.uint64(seed & 0xFFFFFFFF), np.uint64((seed >> 32) & 0xFFFFFFFF)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c0
        p1 = np.uint64(0xCD9E8D57) * c2
        c0, c1, c2, c3 = ((p1 >> np.uint64(32)) ^ c1 ^ k0) & M, p1 & M, ((p0 >> np.uint64(32)) ^ c3 ^ k1) & M, p0 & M
        k0 = (k0 + np.uint64(0x9E3779B9)) & M; k1 = (k1 + np.uint64(0xBB67AE85)) & M
    return ((c0 >> np.uint64(8)).astype(np.float32) * np.float32(1.0 / 16777216.0)).astype(np.float32)


def test_header_declares_and_library_exports_the_windowed_entry_points():
    src = open(os.path.join(ROOT, "include", "nvwn_b200.h")).read()
    lib = _lib.lib()
    for name in NEW:
        assert re.search(rf"\bint {name}\(", src), f"nvwn_b200.h does not declare {name}"
        assert hasattr(lib, name) and name in _lib.SYMBOLS


def test_selector_range_is_the_slice_of_the_whole_draw():
    B, N, seed = 7, 300, 0x5EED0B17C4
    whole = philox_selectors(N * B, seed).reshape(N, B)
    for first, n in ((0, 1), (13, 40), (299, 1), (100, 200)):
        t = np.arange(first, first + n, dtype=np.uint64)[:, None]
        got = philox_at(t * np.uint64(B) + np.arange(B, dtype=np.uint64)[None, :], seed)
        assert np.array_equal(got.view(np.uint32), whole[first:first + n].view(np.uint32))
    # counters past 2^32 (sample indices near 2^31 at B > 2) use the high counter word
    hi = np.uint64(2 ** 31 - 2) * np.uint64(B)
    assert hi > 2 ** 32
    v = philox_at(np.array([hi, hi + np.uint64(1)]), seed)
    assert np.all((v >= 0) & (v < 1)) and v[0] != v[1]
