"""bench.py's JSON contract, exercised on the CPU through the reference arm (`--impl reference` times the reference's
own CPU model, oracle/_ref, on a bounded sample): one JSON line with the keys the driver reads.  And --dump-outputs: what
the timed path computed, written so that two runs or two builds can be compared."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    if not os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libnvwn_ref.so")):
        pytest.skip("oracle/_ref not built")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                          "--cpu-samples", "8", "--batch", "8"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "samples/s" and d["higher_is_better"] is True and d["n_gpus"] == 1
    assert d["steps"] == 2 and d["warmup"] == 1 and d["value"] > 0 and d["ms_per_step"] > 0 and d["vs_baseline"] is None
    assert d["scaling"] == "weak" and d["data"] == "synthetic" and "workload" in d["config"]
    sys.path.insert(0, ROOT)
    import bench
    assert d["metric"] == bench.metric_name() and "fp16" not in d["metric"]      # one metric string for both arms: precision lives in `dtype`
    cb = d["cpu_baseline"]
    assert cb["kind"] == "reference" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    e2e = d["e2e"]
    assert e2e["value"] == d["value"] and e2e["unit"] == d["unit"] and e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0


def test_dump_outputs_keeps_a_fixed_sample_of_utterances_past_the_size_limit(tmp_path):
    sys.path.insert(0, ROOT)
    import bench
    y = np.arange(10 * 6, dtype=np.int32).reshape(10, 6)
    bench.dump_outputs(str(tmp_path / "all"), "yout", y, 10 * 6 * 4)
    whole = np.load(tmp_path / "all" / "yout.npy")
    assert whole.dtype == np.float32 and np.array_equal(whole, y) and not (tmp_path / "all" / "yout_rows.npy").exists()
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), "yout", y, 4 * 6 * 4 + 5)
    rows = np.load(tmp_path / "a" / "yout_rows.npy")
    assert rows.dtype == np.float64 and len(rows) == 4 and np.all(np.diff(rows) > 0)
    assert np.array_equal(np.load(tmp_path / "a" / "yout.npy"), y[rows.astype(int)])
    assert np.array_equal(rows, np.load(tmp_path / "b" / "yout_rows.npy"))


@pytest.mark.gpu
def test_our_arm_dumps_the_same_outputs_from_run_to_run(tmp_path):
    """--dump-outputs writes the last timed step's yOut; with the same arguments two runs sample the same indices."""
    lines = []
    for d in ("a", "b"):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "3", "--warmup", "1", "--samples", "1000",
                              "--no-extra", "--no-cpu", "--no-e2e", "--dump-outputs", str(tmp_path / d)],
                             capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        lines.append(json.loads(out.stdout.strip().splitlines()[-1]))
    assert lines[0]["steps"] == 3 and lines[0]["value"] > 0
    ya, yb = np.load(tmp_path / "a" / "yout.npy"), np.load(tmp_path / "b" / "yout.npy")
    assert ya.dtype == np.float32 and ya.shape == (lines[0]["config"]["batch_per_gpu"], 1000)
    assert ya.min() >= 0 and ya.max() < 256 and len(np.unique(ya)) > 16
    assert np.array_equal(ya, yb)


def test_reference_arm_nonzero_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1",
                          "--cpu-samples", "8", "--batch", "8"], capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""
