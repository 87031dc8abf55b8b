"""The fp16 kernels' softmax and sampling stage when every logit is shifted by the same amount.

Softmax is invariant under a common shift of the logits, so the kernels must be too: P is checked against a float64 softmax
of the kernel's own dumped Za (the exact reference for this stage), with a margin measured on the unshifted logits.  The
CPU oracle cannot serve here at large negative shifts: it starts its row max at 0, like the reference CPU model.
"""
import numpy as np
import pytest

import nv_wavenet_b200 as nw
from oracle import pyoracle as po
from tests import refgen
from tests.test_gpu_parity import _check_sampled_index, _logit_check, _select_fp16_kernel, cpu_oracle, gpu_engine

pytestmark = pytest.mark.gpu

R, S, A, L, B, N, MD = 64, 256, 256, 12, 20, 8, 8              # two 16-utterance tiles, the second one ragged
KERNELS = ["stream", "lat", "lat_single", "tc"]
SHIFTS = [40.0, 0.0, -40.0, -120.0]
EDGE_SELECTORS = np.array([0.0, 2.0 ** -24, 1.0 - 2.0 ** -24, 1.0], np.float32)     # libc-mode selectors can be exactly 1.0


def softmax64(za):
    z = za.astype(np.float64)
    e = np.exp(z - z.max(axis=1, keepdims=True))
    return e / e.sum(axis=1, keepdims=True)


def _inputs(shift, edge_selectors=False):
    w = refgen.lively_inputs(404, R, S, A, L, B, N)
    w["Bza"] = (w["Bza"] + np.float32(shift)).astype(np.float32)
    if edge_selectors:
        w["selectors"] = w["selectors"].copy()
        w["selectors"][:, :len(EDGE_SELECTORS)] = EDGE_SELECTORS
        w["selectors"][:, B - len(EDGE_SELECTORS):] = EDGE_SELECTORS                   # and in the ragged tile
    return w


FORCED = np.random.default_rng(404).integers(0, A, (B, N)).astype(np.int32)


def _run(kernel, w):
    e = gpu_engine(w, L, B, N, R, S, A, MD, dtype=nw.FP16)
    e.set_forced(FORCED)
    y = np.zeros((B, N), np.int32)
    e.run(N, B, y, dump_activations=True); e.synchronize()
    info = e.launch_info()
    assert info["kernel"] == {"stream": 16, "lat": 18, "lat_single": 18}.get(kernel, 17)
    if kernel.startswith("lat"):
        assert info["cluster"] == (3 if kernel == "lat" else 1)
    za, p = e.get_za(), e.get_p()
    e.close()
    return za, p, y[:, N - 1]


def _p_err(za, p):
    return np.abs(p.astype(np.float64) - softmax64(za)).max() / softmax64(za).max()


@pytest.mark.parametrize("shift", SHIFTS)
@pytest.mark.parametrize("kernel", KERNELS)
def test_fp16_softmax_under_logit_shift(kernel, shift, monkeypatch):
    _select_fp16_kernel(kernel, monkeypatch)
    za0, p0, _ = _run(kernel, _inputs(0.0))
    assert np.all(np.isfinite(p0))
    margin = max(2e-3, 2 * _p_err(za0, p0))                    # what the stage achieves on unshifted logits
    w = _inputs(shift)
    za, p, y = _run(kernel, w)
    if shift < 0:
        assert za.max() < 0, "the shift must make every logit negative"
    assert np.all(np.isfinite(p)), f"non-finite P at logit shift {shift}"
    assert np.allclose(p.sum(axis=1), 1.0, atol=1e-3)
    ref = softmax64(za)
    err = _p_err(za, p)
    assert err <= margin, f"|P - softmax(Za)| / max P = {err:.3g} at logit shift {shift}, {margin:.3g} unshifted"
    _check_sampled_index(ref, w["selectors"][N - 1], y)
    if shift >= -40:
        o16 = cpu_oracle(w, L, B, N, R, S, A, MD, prec=po.PREC_FP16); o16.set_forced(FORCED); o16.run(N, B)
        _logit_check(o16.get_za(), za, 1e-2)


@pytest.mark.parametrize("shift", [0.0, -120.0])
@pytest.mark.parametrize("kernel", KERNELS)
def test_fp16_selector_edges(kernel, shift, monkeypatch):
    """Selectors 0, 2^-24, 1 - 2^-24 and 1.0: the sampled class has nonzero probability and follows the cumulative rule."""
    _select_fp16_kernel(kernel, monkeypatch)
    w = _inputs(shift, edge_selectors=True)
    za, p, y = _run(kernel, w)
    ref = softmax64(za)
    _check_sampled_index(ref, w["selectors"][N - 1], y)
    for b in list(range(len(EDGE_SELECTORS))) + list(range(B - len(EDGE_SELECTORS), B)):
        assert ref[b, y[b]] > 0 and p[b, y[b]] > 0, f"utterance {b}: selector {w['selectors'][N - 1, b]} sampled class {y[b]} of probability {p[b, y[b]]}"
