"""Windowed against full engines at the C3 model (L20 R64 S256 A256, maxDilation 512), fp16, AUTO kernel choice.

    python tools/bench_window.py [--reps 5] [--no-long]

1. B = 64, N = 16 000, chunks of 2 000 samples: a full engine (stores for all N samples) and a windowed engine (W = 2 chunks) run
   the SAME pipeline -- mel frames -> conditioning producer on a side stream one chunk ahead (ConvTranspose1d(80, 80, 800, 200),
   1x1 cond layer), per-chunk counter-based selectors, generation, device mu-law decode to int16 -- alternated `reps` times; CUDA
   events around the whole pipeline.  The sampled audio of the two must be identical.
2. Long form: 720 utterances x 160 000 samples through a windowed engine with chunks of 4 000 (W = 8 000).  A full engine of
   this size would need (L x 256 + 12) bytes x 720 x 160 000 = 591 GB.

Prints one JSON line per measurement, with the card's name and power limit.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import nv_wavenet_b200 as nw  # noqa: E402
from tests import refgen  # noqa: E402

L, R, S, A, MD = 20, 64, 256, 256, 512
C_MEL, K_UP, STRIDE = 80, 800, 200
SEED = 20261017


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in out.split(",")]
    except Exception as ex:                              # the numbers are still printed, with what is known about the card
        name, power = torch.cuda.get_device_name(0), f"unknown ({str(ex)[:60]})"
    return {"card": name, "power_limit": power}


def engine(B, n, window):
    w = refgen.lively_inputs(7, R, S, A, L, 1, 1)
    e = nw.NVWavenetInfer(L, MD, B, n, R=R, S=S, A=A, dtype=nw.FP16, window=window)
    e.load(w)
    return e


def mel(B, n):
    g = torch.Generator(device="cuda"); g.manual_seed(SEED)
    rnd = lambda *shape, s=1.0: torch.randn(shape, generator=g, device="cuda", dtype=torch.float32) * s
    return (rnd(B, C_MEL, n // STRIDE), rnd(C_MEL, C_MEL, K_UP, s=0.02), rnd(C_MEL, s=0.01), rnd(L * 2 * R, C_MEL, s=0.05),
            rnd(L * 2 * R, s=0.05))


def pipeline(e, B, n, chunk, windowed, keep=None):
    """The whole utterance batch through `e` in chunks; returns milliseconds (CUDA events) and, with keep, the int16 audio of
    utterances `keep` as a host array."""
    main, side = torch.cuda.current_stream(), torch.cuda.Stream()
    starts = list(range(0, n, chunk))
    out = torch.empty((len(keep), n), dtype=torch.int16, device="cuda") if keep is not None else None
    kidx = torch.as_tensor(keep, device="cuda") if keep is not None else None
    audio = [torch.empty((B, min(chunk, n - s0)), dtype=torch.int16, device="cuda") for s0 in starts[:2]]
    e.reset_history()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record(main)
    side.wait_stream(main)
    produced, decoded = [], []

    def produce(k):
        if windowed and k >= 2:
            side.wait_event(decoded[k - 2])              # chunk k overwrites the slots of chunk k - 2
        e.cond_producer_run(starts[k], min(chunk, n - starts[k]), stream=side)
        ev = torch.cuda.Event(); ev.record(side); produced.append(ev)

    produce(0)
    for k, s0 in enumerate(starts):
        m = min(chunk, n - s0)
        if k + 1 < len(starts):
            produce(k + 1)
        e.set_selectors_random_range(SEED, s0, m, stream=main)
        main.wait_event(produced[k])
        e._samples_per_chunk = m
        e.run_partial(s0, n, B, None, 1, False, main)
        e._samples_per_chunk = 0
        a = audio[k % 2] if m == audio[k % 2].shape[1] else torch.empty((B, m), dtype=torch.int16, device="cuda")
        e.get_audio(s0, m, int16=True, out=a, stream=main)
        if out is not None:
            out[:, s0:s0 + m] = a.index_select(0, kidx)
        ev = torch.cuda.Event(); ev.record(main); decoded.append(ev)
    t1.record(main)
    torch.cuda.synchronize()
    return t0.elapsed_time(t1), (out.cpu().numpy() if out is not None else None)


def compare(reps):
    B, n, chunk = 64, 16000, 2000
    feats = mel(B, n)
    engines = {"full": engine(B, n, None), "windowed": engine(B, None, 2 * chunk)}
    for e in engines.values():
        e.cond_producer_load(*feats, STRIDE)
    audio = {k: pipeline(e, B, n, chunk, k == "windowed", keep=list(range(B)))[1] for k, e in engines.items()}   # warm-up
    assert np.array_equal(audio["full"], audio["windowed"]), "windowed audio differs from the full engine's"
    ms = {k: [] for k in engines}
    for _ in range(reps):
        for k, e in engines.items():
            ms[k].append(pipeline(e, B, n, chunk, k == "windowed")[0])
    info = engines["windowed"].launch_info()
    res = {"case": "C3 B=64 N=16000, producer overlapped, chunks of 2000", "kernel": info["kernel"], "cluster": info["cluster"],
           "window": 2 * chunk, "audio_identical": True, **card()}
    for k, v in ms.items():
        res[k] = {"ms_median": round(statistics.median(v), 2), "ms_min": round(min(v), 2), "ms_max": round(max(v), 2),
                  "Msamples_per_s": round(B * n / statistics.median(v) / 1e3, 3), "ms_all": [round(x, 2) for x in v]}
    res["windowed_over_full"] = round(res["windowed"]["ms_median"] / res["full"]["ms_median"], 4)
    for e in engines.values():
        e.close()
    print(json.dumps(res), flush=True)


def long_form():
    B, n, chunk = 720, 160000, 4000
    feats = mel(B, n)
    e = engine(B, None, 2 * chunk)
    e.cond_producer_load(*feats, STRIDE)
    pipeline(e, B, 4 * chunk, chunk, True)                # warm-up on the first four chunks
    ms, _ = pipeline(e, B, n, chunk, True)
    info = e.launch_info()
    per_sample = L * 256 * B                              # fp16 conditioning; + 12 bytes (selector, forcing, output) on a full
    print(json.dumps({"case": "long form 720 x 160000, producer overlapped, chunks of 4000", "kernel": info["kernel"],
                      "cluster": info["cluster"], "window": 2 * chunk, "ms": round(ms, 1),
                      "Msamples_per_s": round(B * n / ms / 1e3, 3), "kHz_per_utterance": round(n / ms, 2),
                      "full_engine_store_GB": round((per_sample + 12 * B) * n / 1e9, 1),       # engine, 8 (no forcing) on a windowed one
                      "windowed_store_GB": round((per_sample + 8 * B) * 2 * chunk / 1e9, 1),
                      **card()}), flush=True)
    e.close()


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--no-long", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_window.py measures on a CUDA device; none is visible")
    compare(args.reps)
    if not args.no_long:
        long_form()
