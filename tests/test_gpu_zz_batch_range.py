"""fp16 generation across the batch range AUTO serves, up to a history ring larger than 4 GiB.

Each case builds its conditioning on the device from one 16-utterance tile of lively inputs, scaled per tile so that a tile
mix-up is visible, and checks a few chosen tiles three ways:
1. a second engine that holds only those utterances, forced onto the same kernel variant, produces the same free-running yOut
   bit for bit (tiles never interact and the kernels are deterministic);
2. at matched history (teacher forcing), the logits of one tile agree with the fp32 and the fp16-contract CPU oracle, after
   more than one turn of the history ring, and the sampled index follows the cumulative rule;
3. the launch is the kernel AUTO is documented to pick for that batch.
"""
import ctypes as C

import numpy as np
import pytest

import nv_wavenet_b200 as nw
from oracle import pyoracle as po
from tests import refgen
from tests.common import philox_selectors
from tests.test_gpu_parity import _check_sampled_index, _logit_check, cpu_oracle

pytestmark = pytest.mark.gpu

R, S, A = 64, 256, 256
TU_LAT, TU_TC = 16, 64
SEED_SEL = 0x5EED0B17C4
ORACLE_UTT = 8                 # utterances of one tile checked against the CPU oracle (its cost grows with L x N)
CHUNK_BYTES = 1 << 30          # device conditioning is generated and uploaded in pieces of about this size


def lat_ring_bytes(L, maxdil, B):
    """wn_lat_ring_bytes (wn_lat_kernel.cu): (maxDil + 1) x L x 16-utterance tiles x 2048 bytes."""
    return (maxdil + 1) * L * ((B + TU_LAT - 1) // TU_LAT) * 2048


def lat_max_clusters():
    from nv_wavenet_b200 import _lib
    fn = _lib.lib().nvwn_debug_lat_max_clusters
    fn.restype, fn.argtypes = C.c_int, [C.c_int]
    n = fn(S)
    assert n > 0
    return n


def tile_scale(b):
    """Per-utterance factor of the conditioning: 1 + 0.02 * ((b // 16) % 7), in float32."""
    return (1.0 + 0.02 * ((np.asarray(b) // 16) % 7)).astype(np.float32)


def first_wrap_victim(L, maxdil, ntiles):
    """The tile whose history the first wrapped 32-bit ring offset lands on: (slot * L + l) * rstride, rstride = tiles x 2048,
    first passes 2^32 at row k; what is left past 2^32 is a whole number of 2048-byte tiles of row 0, counted from the writer."""
    rs = ntiles * 2048
    k = -(-2 ** 32 // rs)
    assert k < (maxdil + 1) * L
    return ((k * rs - 2 ** 32) // 2048) % ntiles


def host_lh(base, idx):
    """Conditioning of utterances `idx` of the big batch, on the host: [N][L][len(idx)][2R]."""
    idx = np.asarray(idx)
    return np.ascontiguousarray(base["Lh"][:, :, idx % 16, :] * tile_scale(idx)[None, None, :, None])


def upload_device_lh(e, base, idx, N, L):
    """The same conditioning for utterances `idx`, generated with torch on the device a few samples at a time."""
    import torch
    idx = np.asarray(idx)
    lh16 = torch.from_numpy(base["Lh"]).cuda()                                     # [N][L][16][2R]
    gather = torch.from_numpy(idx % 16).cuda()
    scale = torch.from_numpy(tile_scale(idx)).cuda()[None, None, :, None]
    step = max(1, CHUNK_BYTES // (L * len(idx) * 2 * R * 4))
    for t0 in range(0, N, step):
        n = min(step, N - t0)
        chunk = (lh16[t0:t0 + n].index_select(2, gather) * scale).contiguous()
        e.set_conditioning(chunk, t0, n)
        torch.cuda.synchronize()                                                   # a device source is read stream-ordered
        del chunk
    del lh16, gather, scale
    torch.cuda.empty_cache()


def tile_rows(tile, tu, B):
    return list(range(tile * tu, min((tile + 1) * tu, B)))


# batch (a function of the resident cluster count), L, maxDil, N, kernel, cluster, tile size
CASES = {
    # ring 4.34 GiB on the single-CTA latency kernel, one full wave of 148 tiles.  Ring offsets pass 2^32 first at
    # (slot 472, layer 10), which is slot 0 of the tile eight further on; layer 9 (dilation 512) reads slot 0 at t = 512
    "A": (lambda fit: 2368, 30, 512, 640, 18, 1, TU_LAT),
    # ring 5.63 GiB on the three-CTA cluster kernel with every cluster resident (45 on a B200: first wrap at slot 728)
    "B": (lambda fit: 16 * fit, 64, 1024, 1100, 18, 3, TU_LAT),
    # one utterance past the cluster kernel's range: single-CTA kernel, last tile holds one utterance
    "C": (lambda fit: 16 * fit + 1, 12, 64, 100, 18, 1, TU_LAT),
    # one utterance past the latency kernels' range: tensor-core kernel, last 64-utterance tile holds one utterance
    "D": (lambda fit: 2369, 12, 64, 100, 17, 1, TU_TC),
    # tensor-core kernel over more tiles than SMs (two waves), ragged last tile of 24 utterances
    "E": (lambda fit: 9472 + 24, 12, 16, 48, 17, 1, TU_TC),
}


def _clear_env(monkeypatch):
    for k in ("NVWN_FP16_KERNEL", "NVWN_TC_TILE", "NVWN_TC_NODUP", "NVWN_TC_FUSED", "NVWN_LAT_CLUSTER", "NVWN_LAT_MAX_B"):
        monkeypatch.delenv(k, raising=False)


@pytest.mark.parametrize("case", sorted(CASES))
def test_fp16_batch_range(case, monkeypatch):
    import torch
    batch_of, L, md, N, kernel, cluster, tu = CASES[case]
    fit = lat_max_clusters()
    B = batch_of(fit)
    ntiles = (B + tu - 1) // tu
    tiles = [0, ntiles // 2, ntiles - 1]                            # first, middle, last (ragged where B is not a multiple of tu)
    oracle_tile = ntiles // 2
    if case in ("A", "B"):
        assert lat_ring_bytes(L, md, B) > 2 ** 32, "this case exists to put the history ring past 4 GiB"
        assert B <= 2368
        oracle_tile = first_wrap_victim(L, md, ntiles)             # its early history is the first that is overwritten
        tiles = sorted(set(tiles) | {oracle_tile})
    idx = [b for t in tiles for b in tile_rows(t, tu, B)]

    base = refgen.lively_inputs(1000 + B, R, S, A, L, 16, N)
    sel_all = philox_selectors(N * B, SEED_SEL).reshape(N, B)
    forced_all = np.random.default_rng(B).integers(0, A, (B, N)).astype(np.int32)

    # ---- the big engine, AUTO
    _clear_env(monkeypatch)
    e = nw.NVWavenetInfer(L, md, B, N, R=R, S=S, A=A, dtype=nw.FP16)
    e.load(base)
    upload_device_lh(e, base, np.arange(B), N, L)
    e.set_selectors_random(SEED_SEL)
    e.reset_history()
    y_big = np.zeros((B, N), np.int32)
    e.run(N, B, y_big); e.synchronize()
    info = e.launch_info()
    grid = ntiles * cluster if kernel == 18 else ntiles
    assert (info["kernel"], info["cluster"], info["grid"]) == (kernel, cluster, grid), info
    assert len(np.unique(y_big[idx])) > 32
    # ... and teacher-forced, dumping the last step
    e.reset_history(); e.set_forced(forced_all)
    y_f = np.zeros((B, N), np.int32)
    e.run(N, B, y_f, dump_activations=True); e.synchronize()
    za_big, p_big = e.get_za(), e.get_p()
    e.close(); del e
    torch.cuda.empty_cache()

    # ---- 1. the same kernel variant on only the chosen tiles
    if kernel == 17:
        monkeypatch.setenv("NVWN_FP16_KERNEL", "tc")
    else:
        monkeypatch.setenv("NVWN_FP16_KERNEL", "lat")
        if cluster == 1:
            monkeypatch.setenv("NVWN_LAT_CLUSTER", "0")
    es = nw.NVWavenetInfer(L, md, len(idx), N, R=R, S=S, A=A, dtype=nw.FP16)
    es.load(base)
    upload_device_lh(es, base, idx, N, L)
    es.set_selectors(np.ascontiguousarray(sel_all[:, idx]))
    es.reset_history()
    ys = np.zeros((len(idx), N), np.int32)
    es.run(N, len(idx), ys); es.synchronize()
    si = es.launch_info()
    assert (si["kernel"], si["cluster"], si["batch_per_cta"]) == (kernel, cluster, tu), si
    es.close(); del es
    for t in tiles:
        rows = tile_rows(t, tu, B)
        pos = [idx.index(b) for b in rows]
        diff = np.nonzero((ys[pos] != y_big[rows]).any(axis=0))[0]
        assert diff.size == 0, f"tile {t}: yOut differs from the small engine first at sample {diff[:1]} (of {N})"

    # ---- 2. one tile against the CPU oracle at matched history, last step after a full turn of the ring
    assert N - 1 > md + 1
    rows = tile_rows(oracle_tile, tu, B)[:ORACLE_UTT]
    nb = len(rows)
    wo = dict(base); wo["Lh"] = host_lh(base, rows); wo["selectors"] = np.ascontiguousarray(sel_all[:, rows])
    f = np.ascontiguousarray(forced_all[rows])
    za_g, p_g = za_big[rows], p_big[rows]
    o32 = cpu_oracle(wo, L, nb, N, R, S, A, md); o32.set_forced(f); o32.run(N, nb)
    _logit_check(o32.get_za(), za_g, 1e-2)
    o16 = cpu_oracle(wo, L, nb, N, R, S, A, md, prec=po.PREC_FP16); o16.set_forced(f); o16.run(N, nb)
    # the mean tolerance of the 20-layer tests, grown like a random walk over deeper stacks (3.3e-4 measured at L = 64 on a B200)
    _logit_check(o16.get_za(), za_g, 1e-2, mean_rel=3e-4 * max(1.0, np.sqrt(L / 20)))
    assert np.all(np.isfinite(p_g)) and np.allclose(p_g.sum(axis=1), 1.0, atol=1e-3)
    _check_sampled_index(p_g, sel_all[N - 1, rows], y_f[rows, N - 1])
