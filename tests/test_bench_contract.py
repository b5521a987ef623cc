"""bench.py contract checks that run without a GPU: the reference arm prints one JSON line with the
required keys; the ours-arm fails loudly off-GPU instead of falling back."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "1", "--cpu-procs", "2"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
              "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in line, k
    assert line["impl"] == "reference" and line["unit"] == "edges/s" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] in ("port", "reference") and line["cpu_baseline"]["cores"] == 2
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["value"] == line["value"]
    assert "workload" in line["config"] and "model" not in line["config"]


def test_ours_arm_needs_gpu():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("GPU present")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--no-cpu-baseline", "--steps", "1"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode != 0 and "no CPU path" in (out.stderr + out.stdout)


def test_reference_arm_under_torchrun_prints_one_line_from_rank0():
    """N > 1: the driver launches the reference arm with torchrun as well; rank 0 alone measures and prints, and the
    workload is the one the GPU arm defaults to at N > 1 (the Freebase-shaped table, entity count capped and stated)."""
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(29300 + os.getpid() % 500), os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
           "--steps", "1", "--warmup", "1", "--cpu-procs", "2"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, out.stdout[-1000:]
    line = json.loads(lines[0])
    assert line["impl"] == "reference" and line["n_gpus"] == 2 and line["value"] > 0
    assert "Freebase" in line["config"]["workload"] and line["config"]["entities_scaled_down"] is True


def test_dump_outputs_writes_whole_tables_or_a_bounded_sample_of_the_updated_rows(tmp_path, monkeypatch):
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    monkeypatch.setattr(bench, "DUMP_BYTES", 1 << 20)
    g = torch.Generator().manual_seed(0)
    ent, es = torch.randn(5000, 64, generator=g), torch.rand(5000, generator=g)      # 1.3 MB: sampled
    rel, rs = torch.randn(30, 64, generator=g), torch.rand(30, generator=g)          # whole
    ids = torch.randint(0, 5000, (4000,), generator=g)
    log4 = torch.tensor([0.5, 0.25, 0.375, 0.0625])
    tables = {"entity": (ent, es, ids), "relation": (rel, rs, torch.tensor([3, 4]))}
    bench.dump_outputs(str(tmp_path / "a"), log4, tables)
    bench.dump_outputs(str(tmp_path / "b"), log4, tables)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == sorted(["log.npy", "entity_emb.npy", "entity_state.npy", "entity_rows.npy", "relation_emb.npy",
                            "relation_state.npy"])
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= bench.DUMP_BYTES
    z = {f[:-4]: np.load(tmp_path / "a" / f) for f in files}
    for f in files:                                                                  # seeded: the same sample twice
        np.testing.assert_array_equal(z[f[:-4]], np.load(tmp_path / "b" / f))
    assert all(a.dtype in (np.float32, np.float64) for a in z.values())
    rows = z["entity_rows"].astype(np.int64)
    assert z["entity_rows"].dtype == np.float64 and np.all(np.diff(rows) > 0) and set(rows) <= set(ids.tolist())
    np.testing.assert_array_equal(z["entity_emb"], ent[rows].numpy())
    np.testing.assert_array_equal(z["entity_state"], es[rows].numpy())
    np.testing.assert_array_equal(z["relation_emb"], rel.numpy())
    np.testing.assert_array_equal(z["relation_state"], rs.numpy())
    np.testing.assert_array_equal(z["log"], log4.numpy())


@pytest.mark.gpu
def test_bench_dumps_what_its_last_timed_step_computed(tmp_path):
    import numpy as np
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "3", "--warmup", "1", "--no-cpu-baseline",
                          "--no-beside", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == 3 and line["value"] > 0
    z = {f[:-4]: np.load(os.path.join(str(tmp_path), f)) for f in os.listdir(str(tmp_path))}
    assert sorted(z) == ["entity_emb", "entity_state", "log", "relation_emb", "relation_state"]
    assert z["entity_emb"].shape == (14951, 400) and z["relation_emb"].shape == (1345, 400)
    assert all(a.dtype == np.float32 and np.isfinite(a).all() for a in z.values())
    assert z["log"][2] > 0 and (z["entity_state"] > 0).any() and (z["relation_state"] > 0).any()
