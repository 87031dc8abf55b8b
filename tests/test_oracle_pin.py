"""Pins the CPU oracle (oracle/wavenet_oracle.c) to the reference.

1. tests/refgen.py's glibc-rand replay regenerates the reference test's inputs bit-exactly
   (sha256 recorded from the reference's own Matrix::randomize + libc rand()).
2. The oracle in LIBM mode reproduces the reference CPU model bit for bit on all 16 runs of
   the reference integration test (golden vectors made by tests/golden/make_golden.py from
   oracle/_ref = the reference's nv_wavenet_reference.cpp compiled unmodified).
3. The oracle in PORTABLE-math mode (the arithmetic contract the CUDA fp32 kernel implements
   bit-exactly) samples identical indices and stays within a few ulp on activations.
4. The same on fresh shapes/seeds, against the reference CPU model's outputs on them (golden vectors
   made by tests/golden/make_golden.py, as in 2).
"""
import os

import numpy as np
import pytest

from oracle import pyoracle as po
from tests import common, refgen

RUNS = common.reference_runs()
FAST = [r for r in RUNS if r[3] <= 64 and r[5] <= 512]        # R<=64 runs: cheap
ALL_IDS = [r[0] for r in RUNS]


@pytest.mark.parametrize("run", RUNS, ids=ALL_IDS)
def test_refgen_replays_reference_inputs(run):
    key, seed, i, R, S, A, L = run
    w = common.reference_inputs(seed, i)
    assert common.sha([w[k] for k in common.INPUT_KEYS]) == str(common.golden()[key + "/in_sha"])


def _run_oracle(run, math):
    key, seed, i, R, S, A, L = run
    w = common.reference_inputs(seed, i)
    o = po.Oracle(L, common.B_REF, common.N_REF, R, S, A, common.MAXDIL_REF, math=math)
    o.load(w)
    o.set_inputs(w["Lh"], w["selectors"])
    ys, acts = [], []
    for _ in range(common.ITERS_REF):
        ys.append(o.run(common.N_REF, common.B_REF))
        assert o.last_status == 0
        acts.append(o.activations())
    return np.stack(ys), acts


@pytest.mark.parametrize("run", RUNS, ids=ALL_IDS)
def test_oracle_libm_is_bit_exact_vs_reference_cpu(run):
    key = run[0]
    g = common.golden()
    y, acts = _run_oracle(run, po.MATH_LIBM)
    assert np.array_equal(y, g[key + "/y"])
    for it, act in enumerate(acts):
        assert common.sha([act[k] for k in ("xt", "skip", "zs", "za", "p")]) == str(g[key + "/act_sha"][it])


@pytest.mark.parametrize("run", RUNS, ids=ALL_IDS)
def test_oracle_portable_math_same_indices(run):
    key = run[0]
    g = common.golden()
    y, acts = _run_oracle(run, po.MATH_PORTABLE)
    assert np.array_equal(y, g[key + "/y"])                         # exact, as nv_wavenet_test.cu:302-304
    for it, act in enumerate(acts):
        # reference tolerances are 1e-4 (Za) / 1e-3 (p) / 1e-2 (Xout, skip); we hold 2e-6
        assert common.rel_close(g[key + "/za"][it], act["za"], 2e-6, 1e-7)
        assert common.rel_close(g[key + "/p"][it], act["p"], 2e-6)
        assert common.rel_close(g[key + "/xt_last"][it], act["xt"][-1], 2e-6, 1e-7)
        assert common.rel_close(g[key + "/skip_last"][it], act["skip"][-1], 2e-6, 1e-7)


def test_portable_math_accuracy():
    lib = po.Oracle.lib()
    rng = np.random.default_rng(0)
    xs = np.concatenate([rng.uniform(-20, 20, 4000), rng.uniform(-1e-3, 1e-3, 500), [0.0, -0.0, 88.0, -87.0, -100.0, 1e-10]]).astype(np.float32)
    for x in xs:
        e = lib.wno_expf_portable(float(x)); t = lib.wno_tanhf_portable(float(x)); s = lib.wno_sigmoidf_portable(float(x))
        ee = np.exp(np.float64(x)); tt = np.tanh(np.float64(x))
        assert abs(e - ee) <= 0.5000001 * np.spacing(np.float32(ee)) or ee < 1e-37
        assert abs(t - tt) <= 0.5000001 * np.spacing(np.float32(abs(tt))) 
        if abs(x) < 80:      # beyond that expf(-x) overflows in float, as in the reference formula
            assert abs(s - 1 / (1 + np.exp(-np.float64(x)))) <= 4.1 * np.spacing(np.float32(s))
    assert lib.wno_expf_portable(200.0) == np.inf and lib.wno_expf_portable(-200.0) == 0.0
    assert lib.wno_round_fp16(1.0009765625 + 1e-4) == np.float32(np.float16(1.0009765625 + 1e-4))


FRESH_SHAPES = [
    # R, S, A, L, B(max), batch, N, maxDil
    (32, 128, 256, 6, 3, 3, 20, 4),
    (64, 256, 256, 5, 4, 4, 12, 8),       # (the reference CPU model asserts batch_size == max_batch, reference.cpp:72)
    (64, 128, 512, 3, 1, 1, 40, 16),
    (128, 256, 256, 2, 2, 2, 6, 2),
]
FRESH_GENS = ["uniform", "lively"]
FRESH_ITERS = 2
FRESH_GOLDEN = os.path.join(common.HERE, "golden", "reference_cpu_fresh.npz")


def fresh_inputs(shape, gen):
    R, S, A, L, B, bs, N, md = shape
    return (refgen.synthetic_inputs if gen == "uniform" else refgen.lively_inputs)(1234 + R + N, R, S, A, L, B, N)


def fresh_key(shape, gen):
    return "_".join(str(v) for v in shape) + "_" + gen


@pytest.mark.parametrize("shape", FRESH_SHAPES)
@pytest.mark.parametrize("gen", FRESH_GENS)
def test_oracle_vs_reference_cpu_fresh_shapes(shape, gen):
    """Against what the reference CPU model computed on the same inputs (stored by tests/golden/make_golden.py)."""
    R, S, A, L, B, bs, N, md = shape
    w = fresh_inputs(shape, gen)
    key = fresh_key(shape, gen)
    g = np.load(FRESH_GOLDEN)
    assert common.sha([w[k] for k in common.INPUT_KEYS]) == str(g[key + "/in_sha"])
    o = po.Oracle(L, B, N, R, S, A, md, math=po.MATH_LIBM); o.load(w); o.set_inputs(w["Lh"], w["selectors"])
    p = po.Oracle(L, B, N, R, S, A, md, math=po.MATH_PORTABLE); p.load(w); p.set_inputs(w["Lh"], w["selectors"])
    for it in range(FRESH_ITERS):
        yr, yo, yp = g[key + "/y"][it], o.run(N, bs), p.run(N, bs)
        assert np.array_equal(yr, yo)
        ar = {k: g[f"{key}/{k}"][it] for k in ("xt", "skip", "zs", "za", "p")}
        ao, ap = o.activations(), p.activations()
        for k in ar:
            assert common.bits_equal(ar[k][:, :bs], ao[k][:, :bs]) if ar[k].ndim == 3 else common.bits_equal(ar[k][:bs], ao[k][:bs])
        if np.array_equal(yr, yp):
            assert common.rel_close(ar["za"][:bs], ap["za"][:bs], 1e-5, 5e-6)
        else:
            # a selector within float rounding of a CDF edge may legitimately flip one draw (SURVEY.md §4);
            # before the first difference everything must agree
            first = int(np.argmax((yr != yp).any(axis=0)))
            assert np.array_equal(yr[:, :first], yp[:, :first])
            assert first > 0


def test_teacher_forcing_and_trace():
    R, S, A, L, B, N = 32, 128, 256, 3, 2, 10
    w = refgen.lively_inputs(7, R, S, A, L, B, N)
    o = po.Oracle(L, B, N, R, S, A, 4, math=po.MATH_PORTABLE); o.load(w); o.set_inputs(w["Lh"], w["selectors"])
    tr = np.zeros((N, B, A), np.float32); o.set_logit_trace(tr)
    y = o.run(N, B)
    assert np.array_equal(tr[-1], o.get_za())
    # forcing the model's own samples reproduces the free run
    o2 = po.Oracle(L, B, N, R, S, A, 4, math=po.MATH_PORTABLE); o2.load(w); o2.set_inputs(w["Lh"], w["selectors"])
    o2.set_forced(y); tr2 = np.zeros_like(tr); o2.set_logit_trace(tr2)
    assert np.array_equal(o2.run(N, B), y) and np.array_equal(tr, tr2)
    # forcing something else changes later logits but not step 0
    o3 = po.Oracle(L, B, N, R, S, A, 4, math=po.MATH_PORTABLE); o3.load(w); o3.set_inputs(w["Lh"], w["selectors"])
    o3.set_forced((y + 1) % A); tr3 = np.zeros_like(tr); o3.set_logit_trace(tr3); o3.run(N, B)
    assert np.array_equal(tr3[0], tr[0]) and not np.array_equal(tr3[1], tr[1])
