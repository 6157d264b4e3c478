"""The reference arm of bench.py (`--impl reference`) runs without a GPU: the reference's own CPU implementation of the path
(oracle/_ref when the reference compiled here, else the plain-C port) on the host cores, one JSON line with the same metric,
unit and direction as the GPU arm.  This is the one place outside tests/ and smoke() where bench.py may execute oracle/."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    out = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--steps", "2", "--warmup", "1"], cwd=ROOT,
                         capture_output=True, text=True, timeout=600, check=True).stdout
    lines = [l for l in out.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference"
    assert d["metric"] == "audio-seconds synthesized/sec (batched streams)" and d["unit"] == "audio-seconds/s"
    assert d["higher_is_better"] is True and d["steps"] == 2 and d["warmup"] == 1 and d["n_gpus"] == 1
    assert d["value"] > 0 and d["ms_per_step"] > 0
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    e = d["e2e"]
    assert e["value"] == d["value"] and e["unit"] == d["unit"] and e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0
    assert d["config"]["workload"].startswith("config3")
    assert d["vs_baseline"] is None


def test_steps_below_one_are_refused():
    r = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--steps", "0"], cwd=ROOT, capture_output=True, text=True,
                       timeout=120)
    assert r.returncode == 2 and r.stdout == "" and "--steps" in r.stderr, (r.returncode, r.stderr[-300:])


def test_dump_outputs_sample_what_the_rows_hold(tmp_path, monkeypatch):
    """--dump-outputs: the seeded sample of a batch output (here a host tensor) is exactly what the rows hold, zero past each
    row's written count, the same for the same seed, and a sample of whole rows when the output exceeds the budget."""
    import numpy as np
    import torch
    monkeypatch.setenv("NCCL_DEBUG", "WARN")
    monkeypatch.syspath_prepend(ROOT)
    import bench
    rows_n, stride, count = 300, 1008, 1000
    out = np.random.default_rng(5).integers(-32768, 32768, size=(rows_n, stride)).astype(np.int16)
    written = np.full(rows_n, count, dtype=np.int32)
    written[::7] = 500
    got = bench.sample_pcm(torch.from_numpy(out), count, written, 0xB200, points=5000)
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    r, c = (got["points_index"] // count).astype(int), (got["points_index"] % count).astype(int)
    assert len(set(got["points_index"])) == 5000 and (c < count).all()
    np.testing.assert_array_equal(got["points"], np.where(c < written[r], out[r, c], 0))
    sel = got["rows_index"].astype(int)
    assert len(sel) == rows_n  # a small output fits whole
    np.testing.assert_array_equal(got["rows"], np.where(np.arange(count)[None, :] < written[sel][:, None], out[sel, :count], 0))
    np.testing.assert_array_equal(got["written"], written)
    again = bench.sample_pcm(torch.from_numpy(out), count, written, 0xB200, points=5000)
    assert all(np.array_equal(got[k], again[k]) for k in got)
    bench.dump_outputs(str(tmp_path), got)
    assert sorted(os.listdir(tmp_path)) == sorted(k + ".npy" for k in got)
    np.testing.assert_array_equal(np.load(tmp_path / "rows.npy"), got["rows"])
    # an output larger than the budget: whole rows of a sample of the rows, and the total stays within the budget
    monkeypatch.setattr(bench, "DUMP_BYTES", 2_000_000)
    part = bench.sample_pcm(torch.from_numpy(out), count, written, 0xB200, points=5000)
    sel = part["rows_index"].astype(int)
    assert 0 < len(sel) < rows_n and sum(a.nbytes for a in part.values()) <= bench.DUMP_BYTES
    np.testing.assert_array_equal(part["rows"], np.where(np.arange(count)[None, :] < written[sel][:, None], out[sel, :count], 0))


def test_reference_arm_other_ranks_exit_quietly():
    """Under torchrun (N > 1) rank 0 alone runs the reference arm; the other ranks exit 0 without work and without output."""
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT="29533")
    r = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"], cwd=ROOT, env=env,
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and r.stdout.strip() == "", (r.returncode, r.stdout[:200], r.stderr[-300:])
