"""Generates tests/golden/reference_cpu.npz from the reference's OWN CPU model.

Run in the build container (needs /root/reference -> oracle/_ref/libnvwn_ref.so):

    python tests/golden/make_golden.py

For every runTest<>() of the reference integration test (nv_wavenet_test.cu:343-394: seeds
3/10/30/50/70, 16 runs, L=20 (12 for A=1024), batch 16, 8 samples, maxDilation 8, two iterations)
it replays the test's inputs with the reference's own Matrix::randomize + libc rand()
(oracle/ref_shim.cpp: ref_gen_test_inputs), runs nvWavenetReference::run twice, and stores

    <key>/y          int32 [2][B][N]   sampled indices of both iterations
    <key>/in_sha     sha256 of every input array's bytes (weights, Lh, selectors)
    <key>/act_sha    sha256 of the last-sample activations (Xt, skip, Zs, Za, p) per iteration
    <key>/za, /p     float32 [2][B][A] last-sample logits and probabilities
    <key>/xt_last    float32 [2][B][R] last layer output, /skip_last float32 [2][B][S]

Inputs are not stored (tests/refgen.py regenerates them bit-exactly; in_sha proves it).

It also writes reference_cpu_fresh.npz: for the fresh shapes of tests/test_oracle_pin.py (synthetic and lively
inputs, FRESH_ITERS runs each), <key>/in_sha and, per run, <key>/y int32 [batch][N] and the last-sample
activations <key>/xt [L][B][R], /skip [L][B][S], /zs, /za, /p [B][A].
"""
import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import pyoracle as po          # noqa: E402
from tests import refgen                   # noqa: E402

B, N, MAXDIL, ITERS = 16, 8, 8, 2
INPUT_KEYS = ["selectors", "embPrev", "embCur", "Wprev", "Wcur", "Bh", "Wres", "Bres", "Wskip", "Bskip",
              "Wzs", "Bzs", "Wza", "Bza", "Lh"]


def sha(arrs):
    h = hashlib.sha256()
    for a in arrs:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def main():
    po.build()
    out = {}
    for seed, runs in refgen.REFERENCE_TEST_GROUPS:
        for i, (R, S, A, Lo) in enumerate(runs):
            L = Lo or 20
            w = po.ref_gen_test_inputs(seed, R, S, A, L, B, N, reseed=(i == 0))
            ref = po.RefCPU(L, B, N, R, S, A, MAXDIL)
            ref.load(w)
            ref.set_inputs(w["Lh"], w["selectors"])
            key = f"s{seed}_r{i}_R{R}_S{S}_A{A}_L{L}"
            ys, shas, za, p, xt, sk = [], [], [], [], [], []
            for _ in range(ITERS):
                ys.append(ref.run(N, B))
                act = ref.activations()
                shas.append(sha([act[k] for k in ("xt", "skip", "zs", "za", "p")]))
                za.append(act["za"]); p.append(act["p"]); xt.append(act["xt"][-1]); sk.append(act["skip"][-1])
            out[key + "/y"] = np.stack(ys)
            out[key + "/in_sha"] = np.array(sha([w[k] for k in INPUT_KEYS]))
            out[key + "/act_sha"] = np.array(shas)
            out[key + "/za"] = np.stack(za); out[key + "/p"] = np.stack(p)
            out[key + "/xt_last"] = np.stack(xt); out[key + "/skip_last"] = np.stack(sk)
            print(key, "ok")
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_cpu.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


def fresh():
    from tests import test_oracle_pin as pin
    out = {}
    for shape in pin.FRESH_SHAPES:
        R, S, A, L, B, bs, N, md = shape
        for gen in pin.FRESH_GENS:
            w = pin.fresh_inputs(shape, gen)
            ref = po.RefCPU(L, B, N, R, S, A, md)
            ref.load(w)
            ref.set_inputs(w["Lh"], w["selectors"])
            key = pin.fresh_key(shape, gen)
            runs = []
            for _ in range(pin.FRESH_ITERS):
                y = ref.run(N, bs)
                runs.append(dict(ref.activations(), y=y))
            out[key + "/in_sha"] = np.array(sha([w[k] for k in INPUT_KEYS]))
            for k in runs[0]:
                out[f"{key}/{k}"] = np.stack([r[k] for r in runs])
            print(key, "ok")
    np.savez_compressed(pin.FRESH_GOLDEN, **out)
    print("wrote", pin.FRESH_GOLDEN, os.path.getsize(pin.FRESH_GOLDEN), "bytes")


if __name__ == "__main__":
    main()
    fresh()
