"""bench.py's reference arm (the CPU leg the driver runs next to the GPU arm) prints one JSON line with the contract's
keys; runs here without a GPU (bounded sample: 50 queries x the TVR corpus, one step)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                        "--warmup", "1", "--cpu-sample-queries", "50"], cwd=ROOT, capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout[-2000:]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "query-video pairs scored+ranked/sec" and d["unit"] == "pairs/s"
    for k in ("value", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
              "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["higher_is_better"] is True and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert d["config"]["workload"] == "tvr_two_scale" and d["config"]["queries"] == 10895
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["value"] > 0


def test_other_ranks_of_the_reference_arm_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                        "--warmup", "1"], cwd=ROOT, capture_output=True, text=True, timeout=300, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_reference_arm_frame_head_times_the_unmodified_reference():
    """--workload tvr_frame: the head the reference ships is timed on the UNMODIFIED reference (baseline/_ref, staged
    by oracle/install_ref.py), kind "reference"."""
    import pytest
    from oracle import install_ref
    install_ref.install()
    if not install_ref.staged():
        pytest.skip("the original DL-DKD sources are not present to stage (they are not part of this repository)")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "tvr_frame",
                        "--steps", "1", "--warmup", "1", "--cpu-sample-queries", "50"], cwd=ROOT, capture_output=True,
                       text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.strip()][-1])
    assert d["impl"] == "reference" and d["config"]["workload"] == "tvr_frame"
    assert d["cpu_baseline"]["kind"] == "reference" and "baseline/_ref" in d["cpu_baseline"]["sample"]
    assert d["value"] > 0 and d["e2e"]["h2d_bytes_per_step"] == 0


def test_dump_outputs_writes_float_arrays_within_the_budget(tmp_path, monkeypatch):
    """--dump-outputs: floating point arrays as float32, integer arrays as float64 (exact); above the byte budget
    every array keeps the same fixed, seeded fraction of its rows (listed in <name>_rows.npy; arrays with as many rows
    keep the same rows), whatever their leading dimensions, and scalars are kept."""
    import numpy as np
    import torch
    import bench
    s = torch.randn(300, 100, generator=torch.Generator().manual_seed(0))
    i = torch.arange(30000, dtype=torch.int32).reshape(300, 100)
    c = torch.randn(40, 8, 100, generator=torch.Generator().manual_seed(1))
    loss = torch.tensor(1.5)
    bench.dump_outputs(str(tmp_path / "full"), {"top_scores": s, "top_ids": i})
    assert sorted(p.name for p in (tmp_path / "full").iterdir()) == ["top_ids.npy", "top_scores.npy"]
    a, b = np.load(tmp_path / "full" / "top_scores.npy"), np.load(tmp_path / "full" / "top_ids.npy")
    assert a.dtype == np.float32 and np.array_equal(a, s.numpy())
    assert b.dtype == np.float64 and np.array_equal(b, i.numpy())
    monkeypatch.setattr(bench, "DUMP_BYTES", 100_000)
    arrays = {"top_scores": s, "top_ids": i, "grad_ctx": c, "loss": loss}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    got = [{p.name[:-4]: np.load(p) for p in (tmp_path / d).iterdir()} for d in ("a", "b")]
    assert sorted(got[0]) == ["grad_ctx", "grad_ctx_rows", "loss", "top_ids", "top_ids_rows", "top_scores",
                              "top_scores_rows"]
    assert sum(x.nbytes for x in got[0].values()) <= 100_000
    assert got[0]["loss"].shape == () and float(got[0]["loss"]) == 1.5
    for name in ("top_scores", "top_ids", "grad_ctx"):
        rows = got[0][name + "_rows"].astype(np.int64)
        assert len(rows) > 0 and np.array_equal(rows, np.unique(rows))
        assert np.array_equal(got[0][name], arrays[name].double().numpy()[rows].astype(got[0][name].dtype))
    assert np.array_equal(got[0]["top_scores_rows"], got[0]["top_ids_rows"])
    assert all(np.array_equal(got[0][k], got[1][k]) for k in got[0])
