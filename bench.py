#!/usr/bin/env python
"""bench.py -- headline benchmark of the WaveNet inference hot path (contract: see DESIGN.md §7).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[2], "C3"): fp16, 20 layers, R64/S256/A256, maxDilation 512,
batch 64 utterances per GPU, 16000 samples per utterance, synthetic conditioning, random weights.
A step = one pass of the hot path: generate all `samples` samples for the whole batch from silence.
metric  = samples/s = (kHz per utterance x batch), whole job over all GPUs   (nv_wavenet_perf.cu:87 x batch)
value   = device-timed (CUDA events on the launch stream), inputs resident in HBM
e2e     = same metric through the public C-ABI with HOST buffers: pinned-host conditioning (fp32, as the
          reference API takes it) uploaded + converted chunk by chunk, overlapped with generation,
          yOut copied back to the host, all inside the timed region
roofline= BASELINE.md §2 normalisation: every utterance-sample is charged one read of all weights+biases
          (+ its Lh, embedding rows, selector, yOut) against the measured HBM copy bandwidth
cpu_baseline / --impl reference = the reference's own CPU model (oracle/_ref, compiled unmodified) on the
          host cores, one process per core, each on a batch shard of the same workload (bounded sample).
"""
import argparse
import json
import multiprocessing as mp
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# BASELINE.json configs: C3 = configs[2] (the headline the metric is quoted on), C2 = configs[1], C4 = configs[3]
CONFIGS = {
    "C3": dict(L=20, R=64, S=256, A=256, max_dilation=512, batch=64, dtype="fp16"),
    "C2": dict(L=20, R=64, S=128, A=256, max_dilation=512, batch=8, dtype="fp16"),
    "C4": dict(L=30, R=128, S=256, A=256, max_dilation=512, batch=16, dtype="fp32"),
}
MODEL = dict(CONFIGS["C3"])
SEED = 20260922


def metric_name():
    """One string for both arms (the driver divides the two lines only if it is identical); precision is in `dtype`."""
    return f"samples/s (kHz/utterance x batch) {MODEL['L']}L R{MODEL['R']}/S{MODEL['S']}/A{MODEL['A']}"


def weight_bytes(L, R, S, A, T):
    return T * (L * (2 * 2 * R * R + R * R + S * R + 3 * R + S) + A * S + A * A + 2 * A)


def algorithmic_bytes(L, R, S, A, T):
    """per utterance-sample (BASELINE.md §2)"""
    return weight_bytes(L, R, S, A, T) + L * 2 * R * T + 2 * R * T + 4 + 4


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def model_weights(seed, L, R, S, A):
    """Random weights with the reference test's distributions (SURVEY.md §8d), numpy fp32, column-major."""
    import numpy as np
    g = np.random.Generator(np.random.PCG64(seed))

    def n(shape, std):
        return (g.standard_normal(shape, dtype=np.float32) * np.float32(std)).astype(np.float32)
    return {
        "embPrev": n((A, R), 0.7), "embCur": n((A, R), 0.7),
        "Wprev": n((L, 2 * R * R), 0.7 / R ** 0.5), "Wcur": n((L, 2 * R * R), 0.7 / R ** 0.5), "Bh": n((L, 2 * R), 0.1),
        "Wres": n((L, R * R), 0.5 / R ** 0.5), "Bres": n((L, R), 0.05),
        "Wskip": n((L, S * R), 0.5 / R ** 0.5), "Bskip": n((L, S), 0.05),
        "Wzs": n(A * S, 1.0 / S ** 0.5), "Bzs": n(A, 0.1), "Wza": n(A * A, 2.0 / A ** 0.5), "Bza": n(A, 0.1),
    }


# --------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.rows, self.proc, self.device = [], None, device

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.device)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------- reference (CPU) arm
def _cpu_worker(args):
    shard_b, n_samples, seed, model = args
    import numpy as np
    from oracle import pyoracle as po
    L, R, S, A, md = model["L"], model["R"], model["S"], model["A"], model["max_dilation"]
    w = model_weights(SEED, L, R, S, A)
    g = np.random.Generator(np.random.PCG64(seed))
    Lh = (g.standard_normal((n_samples, L, shard_b, 2 * R), dtype=np.float32) * np.float32(0.5))
    sel = g.random((n_samples, shard_b), dtype=np.float32)
    ref = po.RefCPU(L, shard_b, n_samples, R, S, A, md)
    ref.load(w)
    ref.set_inputs(Lh, sel)
    t0 = time.perf_counter()
    ref.run(n_samples, shard_b)
    return time.perf_counter() - t0


def cpu_reference_rate(batch, n_samples, cores=None):
    """samples/s of the reference's own CPU model (oracle/_ref) on `cores` host cores: one process per core,
    each generating n_samples samples for its batch shard.  Returns (rate, cores_used, wall_s)."""
    from oracle import pyoracle as po
    if not po.have_ref():
        po.build()
    kind = "reference" if po.have_ref() else "port"
    if kind != "reference":
        raise RuntimeError("oracle/_ref missing")
    cores = cores or os.cpu_count() or 1
    procs = max(1, min(cores, batch))
    shards = [batch // procs + (1 if i < batch % procs else 0) for i in range(procs)]
    ctx = mp.get_context("fork")
    with ctx.Pool(procs) as pool:
        t0 = time.perf_counter()
        times = pool.map(_cpu_worker, [(b, n_samples, 1000 + i, MODEL) for i, b in enumerate(shards)])
        wall = time.perf_counter() - t0
    return batch * n_samples / max(times), procs, wall, kind


def run_reference(args, rank, world):
    if rank != 0:
        return
    batch = args.batch * args.gpus
    n = args.cpu_samples
    for _ in range(max(0, args.warmup - 2)):           # CPU needs no GPU-style warm-up; one pass pages the code in
        cpu_reference_rate(batch, max(2, n // 8))
    rates, cores = [], 1
    t0 = time.perf_counter()
    for _ in range(args.steps):
        r, cores, wall, kind = cpu_reference_rate(batch, n)
        rates.append(r)
    ms = (time.perf_counter() - t0) * 1e3 / args.steps
    value = statistics.mean(rates)
    line = {
        "impl": "reference", "metric": metric_name(), "value": value, "unit": "samples/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, batch),
        "cpu_baseline": {"value": value, "unit": "samples/s", "cores": cores, "kind": kind,
                         "sample": f"nv_wavenet_reference.cpp (unmodified, -O2), {cores} processes x batch shard of {batch}, {n} samples each"},
        "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def workload_config(args, batch):
    return {"workload": f"{args.config}: WaveNet autoregressive inference, {MODEL['L']} layers R{MODEL['R']}/S{MODEL['S']}/A{MODEL['A']} "
                        f"maxDilation{MODEL['max_dilation']}, batch {args.batch}/GPU ({batch} total) x {args.samples} samples",
            "weights": "random N(0, sigma) per matrix (lively gates), not the reference test's U(-0.25/R, 0.25/R): no effect on speed",
            "batch_per_gpu": args.batch, "global_batch": batch, "samples_per_utterance": args.samples,
            "parallelism": f"batch-shard x{args.gpus} (no per-step collective)",
            "l2_policy": "conditioning stream (>5 GB/step) exceeds L2; weights are L2/SMEM-resident by design",
            **({"note": os.environ["NVWN_BENCH_NOTE"]} if os.environ.get("NVWN_BENCH_NOTE") else {})}


# --------------------------------------------------------------------------- extras (single-GPU runs only)
def batch_sweep(nw, torch, args, dtype, T, peak, alg, n_samples=4000):
    """Kernel-only rate at 1x, 2x, 4x the configured batch (same model, shorter utterances): where the normalised roofline
    fraction crosses 0.6 is driver-observable."""
    import numpy as np
    L, R, S, A, md = MODEL["L"], MODEL["R"], MODEL["S"], MODEL["A"], MODEL["max_dilation"]
    w = model_weights(SEED, L, R, S, A)
    out = []
    for mult in (1, 2, 4):
        B = args.batch * mult
        eng = nw.NVWavenetInfer(L, md, B, n_samples, R=R, S=S, A=A, dtype=dtype)
        eng.load(w)
        gen = torch.Generator(device="cuda"); gen.manual_seed(SEED + B)
        chunk = max(1, min(n_samples, (256 << 20) // (L * B * 2 * R * 4)))
        for s0 in range(0, n_samples, chunk):
            n = min(chunk, n_samples - s0)
            eng.set_conditioning(torch.randn((n, L, B, 2 * R), generator=gen, device="cuda", dtype=torch.float32) * 0.5, s0, n)
        eng.set_selectors(torch.rand((n_samples, B), generator=gen, device="cuda", dtype=torch.float32))
        best = None
        for _ in range(3):
            eng.reset_history()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); eng.run(n_samples, B, None); e1.record(); torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            best = ms if best is None else min(best, ms)
        rate = B * n_samples / (best * 1e-3)
        out.append({"batch": B, "samples": n_samples, "khz_per_utterance": n_samples / best, "samples_per_s": rate,
                    "roofline_frac": rate * alg / 1e9 / peak, "kernel": eng.launch_info()["kernel"], "grid": eng.launch_info()["grid"]})
        eng.close()
    return out


def conditioning_producer_timing(eng, torch, args, T):
    """SURVEY.md 8f next-2: mel frames -> upsampling ConvTranspose1d(80, 80, 800, 200) -> 1x1 cond_layers -> the engine's conditioning
    store, on the device (nvwn_set_conditioning_from_features), for the whole utterance batch of this run; one-off per batch."""
    L, R = MODEL["L"], MODEL["R"]
    B, N = args.batch, args.samples
    C, window, stride = 80, 800, 200                         # pytorch/config.json of the reference
    frames = N // stride
    if frames < 1:
        return None
    g = torch.Generator(device="cuda"); g.manual_seed(SEED + 5)
    rnd = lambda *shape, s=1.0: torch.randn(shape, generator=g, device="cuda", dtype=torch.float32) * s
    feats, wu, bu = rnd(B, C, frames), rnd(C, C, window, s=0.02), rnd(C, s=0.01)
    wc, bc = rnd(L * 2 * R, C, s=0.05), rnd(L * 2 * R, s=0.05)
    best = None
    for _ in range(2):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        eng.set_conditioning_from_features(feats, wu, bu, wc, bc, stride)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    out_bytes = frames * stride * L * B * 2 * R * T
    res = {"ms": best * 1e3, "samples": frames * stride, "batch": B, "mel_channels": C, "window": window, "stride": stride,
           "store_GB": out_bytes / 1e9, "store_GB_per_s": out_bytes / 1e9 / best}
    # overlapped: the producer fills the store chunk by chunk on a side stream (nvwn_cond_producer_load / _run) while the main stream
    # generates every chunk as soon as its conditioning is there; against generation alone in the same chunking
    try:
        Ns, chunk = frames * stride, 2000
        main, side = torch.cuda.current_stream(), torch.cuda.Stream()
        eng.cond_producer_load(feats, wu, bu, wc, bc, stride)

        def pipeline(produce):
            eng.reset_history()
            torch.cuda.synchronize()
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record(main)
            evs = []
            if produce:
                side.wait_stream(main)
                for s0 in range(0, Ns, chunk):
                    eng.cond_producer_run(s0, min(chunk, Ns - s0), stream=side)
                    ev = torch.cuda.Event(); ev.record(side); evs.append(ev)
            for i, s0 in enumerate(range(0, Ns, chunk)):
                if produce:
                    main.wait_event(evs[i])
                eng._samples_per_chunk = min(chunk, Ns - s0)
                eng.run_partial(s0, Ns, B, None, 1, False, main)
            eng._samples_per_chunk = 0
            t1.record(main)
            torch.cuda.synchronize()
            return t0.elapsed_time(t1)

        pipeline(True)
        gen_ms, both_ms = min(pipeline(False) for _ in range(2)), min(pipeline(True) for _ in range(2))
        res.update({"overlapped": {"chunk_samples": chunk, "generation_only_ms": gen_ms, "producer_and_generation_ms": both_ms,
                                   "overhead_of_producing_while_generating": both_ms / gen_ms - 1.0}})
    except Exception as ex:                                                    # an extra: never fails the bench line
        res["overlapped"] = {"error": str(ex)[:200]}
    return res


def reference_gpu_kernels(args, our_khz, n_samples=600):
    """The reference's OWN CUDA kernels (oracle/_ref/ref_gpu_harness: unmodified nv_wavenet.cuh rebuilt for sm_100a), same model,
    same batch, same box, timed like nv_wavenet_perf.cu:67-87 -- the GPU baseline next to the headline.  Test infrastructure:
    a separate process; nothing of it is on our path."""
    try:
        from oracle import ref_gpu
        if not ref_gpu.available():
            return {"unavailable": "oracle/_ref/ref_gpu_harness not built"}
        import numpy as np
        L, R, S, A, md = MODEL["L"], MODEL["R"], MODEL["S"], MODEL["A"], MODEL["max_dilation"]
        w = model_weights(SEED, L, R, S, A)
        for k in w:                                     # the reference accumulates in fp16: keep its arithmetic finite
            w[k] = (w[k] * np.float32(0.5)).astype(np.float32)
        g = np.random.Generator(np.random.PCG64(SEED))
        B = args.batch
        w["Lh"] = (g.standard_normal((n_samples, L, B, 2 * R), dtype=np.float32) * np.float32(0.25))
        w["selectors"] = g.random((n_samples, B), dtype=np.float32)
        prec = 16 if args.dtype == "fp16" else 32
        out = {"samples": n_samples, "batch": B, "ours_khz_per_utterance": our_khz}
        best = 0.0
        for mode, name in ((1, "single_block"), (2, "dual_block"), (3, "persistent"), (4, "manyblock")):
            try:
                r = ref_gpu.run(w, prec, R, S, A, L, md, B, n_samples, mode=mode, chunk=2048, reps=2, timeout=120)
                out[name] = {"khz_per_utterance": r["khz"], "samples_per_s": r["samples_per_s"]}
                best = max(best, r["khz"])
            except Exception as ex:       # noqa: BLE001
                out[name] = {"error": str(ex).strip()[-160:]}
        out["best_reference_khz_per_utterance"] = best or None
        out["ours_over_best_reference"] = (our_khz / best) if best else None
        return out
    except Exception as ex:               # noqa: BLE001
        return {"unavailable": str(ex)[:200]}


def dump_outputs(out_dir, name, y, max_bytes):
    """Writes the sampled indices y [utterances][samples] as out_dir/<name>.npy in float32 (exact below 2**24).  When that
    exceeds max_bytes, only a fixed, seeded sample of whole utterances is written, and their indices as <name>_rows.npy."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    keep = max(1, max_bytes // (4 * y.shape[1]))
    if keep < y.shape[0]:
        rows = np.sort(np.random.Generator(np.random.PCG64(SEED)).choice(y.shape[0], keep, replace=False))
        y = y[rows]
        np.save(os.path.join(out_dir, name + "_rows.npy"), rows.astype(np.float64))
    np.save(os.path.join(out_dir, name + ".npy"), y.astype(np.float32))


# --------------------------------------------------------------------------- our arm
def run_ours(args, rank, world, local_rank):
    import numpy as np
    import torch
    import nv_wavenet_b200 as nw

    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    L, R, S, A, md = MODEL["L"], MODEL["R"], MODEL["S"], MODEL["A"], MODEL["max_dilation"]
    B, N = args.batch, args.samples
    dtype = {"fp16": nw.FP16, "fp32": nw.FP32, "fp32fast": nw.FP32_FAST}[args.dtype]
    T = 2 if dtype == nw.FP16 else 4
    eng = nw.NVWavenetInfer(L, md, B, N, R=R, S=S, A=A, dtype=dtype)

    # weights: rank 0 uploads, everyone else receives the packed blob with ONE NCCL broadcast over NVLink
    if rank == 0:
        eng.load(model_weights(SEED, L, R, S, A))
    if world > 1:
        ptr, nbytes = eng.weight_blob()

        class _Blob:
            __cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 3}
        blob = torch.as_tensor(_Blob(), device=torch.device("cuda", local_rank))
        dist.broadcast(blob, 0)
        eng.weights_updated()

    stream = torch.cuda.current_stream()
    # ---- every rank must hold rank 0's weights: all ranks generate the SAME short input (rank 0's seed), run it, and the
    # CRCs of the sampled indices are compared (a rank on a zero / stale blob would run at the same speed but sample differently)
    import zlib
    V = min(N, 256)
    gen0 = torch.Generator(device="cuda"); gen0.manual_seed(SEED)
    eng.set_conditioning(torch.randn((V, L, B, 2 * R), generator=gen0, device="cuda", dtype=torch.float32) * 0.5, 0, V)
    eng.set_selectors(torch.rand((N, B), generator=gen0, device="cuda", dtype=torch.float32))
    eng.reset_history()
    eng._samples_per_chunk = V
    eng.run_partial(0, N, B, None, 1, False, stream)
    eng._samples_per_chunk = 0
    yv = np.zeros((B, N), np.int32)
    eng.get_yout(yv, 0, V, stream); torch.cuda.synchronize()
    crc = zlib.crc32(np.ascontiguousarray(yv[:, :V]).tobytes())
    crcs = [crc]
    if dist:
        tcrc = torch.tensor([crc], device="cuda", dtype=torch.int64)
        allc = [torch.zeros_like(tcrc) for _ in range(world)]
        dist.all_gather(allc, tcrc)
        crcs = [int(c.item()) for c in allc]
    verify = {"yout_crc_equal_across_ranks": len(set(crcs)) == 1, "yout_crc": [f"{c:08x}" for c in crcs], "samples": V,
              "distinct_indices": int(len(np.unique(yv[:, :V])))}
    if not verify["yout_crc_equal_across_ranks"]:
        raise RuntimeError(f"ranks disagree on the same input (weight broadcast broken?): {verify}")

    # synthetic conditioning generated on the device, chunk by chunk, in the kernel's dtype via the public setter
    gen = torch.Generator(device="cuda"); gen.manual_seed(SEED + 17 * rank)
    chunk = max(1, min(N, (256 << 20) // (L * B * 2 * R * 4)))
    for s0 in range(0, N, chunk):
        n = min(chunk, N - s0)
        lh = torch.randn((n, L, B, 2 * R), generator=gen, device="cuda", dtype=torch.float32) * 0.5
        eng.set_conditioning(lh, s0, n)
    torch.cuda.synchronize()
    del lh
    sel = torch.rand((N, B), generator=gen, device="cuda", dtype=torch.float32)
    eng.set_selectors(sel)
    y_dev = torch.zeros((B, N), dtype=torch.int32, device="cuda")

    def step():
        eng.reset_history()
        eng.run(N, B, None, dump_activations=False, stream=stream)

    def barrier():
        torch.cuda.synchronize()
        if dist:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    l0 = eng.launch_info()["launches"] if args.warmup else 0
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    ev0.record(stream)
    for i in range(args.steps):
        eng.reset_history()
        kev[i][0].record(stream)
        eng.run(N, B, None, dump_activations=False, stream=stream)
        kev[i][1].record(stream)
    ev1.record(stream)
    barrier()
    clk = clocks.stop() if rank == 0 else None
    if args.dump_outputs:                   # before the e2e leg below overwrites the conditioning the timed steps ran on
        y = np.zeros((B, N), np.int32)
        eng.get_yout(y, 0, N, stream); torch.cuda.synchronize()
        dump_outputs(args.dump_outputs, "yout" if world == 1 else f"yout_rank{rank}", y, (64 << 20) // world)
    elapsed_ms = ev0.elapsed_time(ev1)
    kernel_ms = statistics.mean(a.elapsed_time(b) for a, b in kev)
    info = eng.launch_info()
    launches = (info["launches"] - l0) + 2 * args.steps          # main kernel + the two history-reset fills per step
    if dist:
        t = torch.tensor([elapsed_ms, kernel_ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed_ms, kernel_ms = t.tolist()
    total_units = world * B * N * args.steps
    value = total_units / (elapsed_ms * 1e-3)

    # ---- e2e through the C-ABI with host buffers (pinned fp32 conditioning, chunked + overlapped) ----
    e2e = None
    if not args.no_e2e:
        e2e_chunk = min(N, args.e2e_chunk)
        host_lh = torch.empty((e2e_chunk, L, B, 2 * R), dtype=torch.float32).pin_memory()
        host_lh.copy_(torch.randn((e2e_chunk, L, B, 2 * R), generator=gen, device="cuda") * 0.5)
        host_sel = torch.empty((N, B), dtype=torch.float32).pin_memory(); host_sel.copy_(sel)
        host_y = torch.empty((B, N), dtype=torch.int32).pin_memory()
        copy_s, out_s = torch.cuda.Stream(), torch.cuda.Stream()

        def e2e_step():
            eng.reset_history()
            eng.set_selectors(host_sel)
            for s0 in range(0, N, e2e_chunk):
                n = min(e2e_chunk, N - s0)
                eng.set_conditioning(host_lh[:n], s0, n, stream=copy_s)          # H2D + fp32->fp16 on the copy stream
                up = torch.cuda.Event(); up.record(copy_s)
                stream.wait_event(up)
                eng._samples_per_chunk = n
                eng.run_partial(s0, N, B, None, 1, False, stream)
                done = torch.cuda.Event(); done.record(stream)
                out_s.wait_event(done)
                eng.get_yout(host_y, s0, n, out_s)                               # D2H of the finished chunk
            eng._samples_per_chunk = 0
            out_s.synchronize()

        e2e_step()
        barrier()
        reps = max(1, min(args.steps, 3))
        t0 = time.perf_counter()
        for _ in range(reps):
            e2e_step()
        torch.cuda.synchronize()
        e2e_s = time.perf_counter() - t0
        if dist:
            t = torch.tensor([e2e_s], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            e2e_s = t.item()
        e2e = {"value": world * B * N * reps / e2e_s, "unit": "samples/s",
               "h2d_bytes_per_step": int(N * L * B * 2 * R * 4 + N * B * 4) * world, "d2h_bytes_per_step": int(B * N * 4) * world,
               "steps": reps, "chunk_samples": e2e_chunk}

    if rank != 0:
        if dist:
            dist.destroy_process_group()
        return

    peak, peak_src = measured_peaks()
    alg = algorithmic_bytes(L, R, S, A, T)
    achieved = B * N * alg / (kernel_ms * 1e-3) / 1e9                # one launch = one step of one GPU
    # DRAM traffic cannot be measured on this run (no profiler in a timed run): `traffic` is dram read + written of the committed
    # `ncu --set full` capture (profiles/ncu_summary.json) when that capture is of exactly this launch (same config, kernel, batch and
    # sample count), else null; `traffic_extrapolated` scales the capture's bytes per unit to this launch in any case
    kname = {16: "wn_stream_kernel", 17: "wn_tc_kernel", 18: "wn_lat2_kernel" if info["cluster"] > 1 else "wn_lat_kernel"}.get(info["kernel"], str(info["kernel"]))
    traffic = None                                  # DRAM bytes of one launch of this very shape, if the committed ncu capture is of it
    traffic_x = None
    prof = os.path.join(ROOT, "profiles", "ncu_summary.json")
    if os.path.exists(prof):
        try:
            pj = json.load(open(prof))
            if pj.get("config") == args.config and pj.get("kernel_id") == info["kernel"] and kname in pj.get("kernel", ""):
                if pj.get("capture_samples") == N and pj.get("capture_batch") == B:
                    traffic = pj["dram_bytes_read"] + pj["dram_bytes_write"]
                traffic_x = {"value": pj["dram_bytes_per_unit"] * B * N, "dram_bytes_per_unit": pj["dram_bytes_per_unit"],
                             "capture_samples": pj.get("capture_samples"), "capture_batch": pj.get("capture_batch"), "source": "profiles/ncu_summary.json"}
        except Exception:
            traffic_x = None
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "traffic_extrapolated": traffic_x, "peak_source": peak_src, "kernel": kname,
                "kernel_ms_per_launch": kernel_ms, "algorithmic_bytes_per_unit": alg, "units_per_launch": B * N,
                "note": "BASELINE.md §2 normalisation: one read of all weights per utterance-sample; weights are re-used across the batch "
                        "on chip, so frac may exceed 1 -- real DRAM traffic is `traffic`"}
    cpu = None
    if not args.no_cpu:
        try:
            r, cores, wall, kind = cpu_reference_rate(B, args.cpu_samples)
            cpu = {"value": r, "unit": "samples/s", "cores": cores, "kind": kind,
                   "sample": f"nv_wavenet_reference.cpp (unmodified, -O2): batch {B} sharded over {cores} processes, {args.cpu_samples} samples each ({wall:.1f}s wall)"}
        except Exception as ex:       # noqa: BLE001
            cpu = {"value": None, "unit": "samples/s", "cores": 0, "kind": "reference", "sample": f"unavailable: {ex}"}
    extra = {"verify": verify}
    if world == 1 and not args.no_extra:
        extra["batch_sweep"] = batch_sweep(nw, torch, args, dtype, T, peak, alg)
        extra["reference_gpu_kernels"] = reference_gpu_kernels(args, N / (elapsed_ms / args.steps))
        extra["conditioning_producer"] = conditioning_producer_timing(eng, torch, args, T)
    line = {
        "metric": metric_name(), "value": value, "unit": "samples/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": elapsed_ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16" if dtype == nw.FP16 else "f32", "arithmetic": {nw.FP16: "fp16 inputs, fp32 accumulate", nw.FP32: "fp32, bit-exact to the reference CPU model", nw.FP32_FAST: "fp32, reference GPU kernels' order (FMA, 2 partial sums)"}[dtype],
        "data": "synthetic", "config": workload_config(args, world * B),
        "khz_per_utterance": N / (elapsed_ms / args.steps), "clocks": clk, "e2e": e2e, "gpu_launches": launches,
        "launch": {k: info[k] for k in ("kernel", "grid", "block", "smem_bytes", "batch_per_cta", "cluster")},
        "roofline": roofline, "cpu_baseline": cpu, "extra": extra,
    }
    print(json.dumps(line), flush=True)
    if dist:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="C3", choices=sorted(CONFIGS), help="BASELINE.json configuration (C3 = headline)")
    ap.add_argument("--batch", type=int, default=None, help="utterances per GPU (default: the configuration's)")
    ap.add_argument("--samples", type=int, default=16000)
    ap.add_argument("--dtype", default=None, choices=["fp16", "fp32", "fp32fast"])
    ap.add_argument("--no-extra", action="store_true", help="skip the batch sweep and the reference-GPU-kernel runs")
    ap.add_argument("--cpu-samples", type=int, default=96, help="samples per utterance of the bounded CPU-reference leg")
    ap.add_argument("--e2e-chunk", type=int, default=1000)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last step's sampled indices (yOut) as DIR/yout.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    MODEL.clear(); MODEL.update(CONFIGS[args.config])
    if args.batch is None:
        args.batch = MODEL["batch"]
    if args.dtype is None:
        args.dtype = MODEL["dtype"]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world != args.gpus and world == 1 and args.gpus > 1:
        # convenience: python bench.py --gpus N re-launches itself under torchrun
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29511", os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    # a device-side failure (the kernels' bounded mbarrier waits trap instead of hanging) is fatal: rc != 0, no re-measurement
    run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
