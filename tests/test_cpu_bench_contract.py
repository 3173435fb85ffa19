"""bench.py contract checks that need no GPU: the reference arm (`--impl reference`, the oracle port on the host cores)
prints one JSON line with the keys the driver reads, and rank > 0 under a multi-rank launch exits without work."""
import json
import os
import subprocess
import sys

from util import ROOT


def _run(args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, env=e, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    return [l for l in p.stdout.strip().splitlines() if l.startswith("{")]


def test_reference_arm_prints_contract_line():
    lines = _run(["--impl", "reference", "--workload", "tiny", "--steps", "1", "--warmup", "0"])
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["n_gpus"] == 1 and d["gpu_launches"] == 0
    for k in ("metric", "value", "unit", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data", "config", "e2e",
              "cpu_baseline"):
        assert k in d, k
    assert d["unit"] == "samples/s" and d["value"] > 0 and d["vs_baseline"] is None
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "utterance" in cb["sample"]
    assert "workload" in d["config"]


def test_dump_outputs_writes_float32_and_samples_whole_rows_over_budget(tmp_path, monkeypatch):
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    wav = torch.arange(6 * 10, dtype=torch.float32).view(6, 10)
    bench.dump_outputs(str(tmp_path / "all"), {"wav": wav})
    a = np.load(tmp_path / "all" / "wav.npy")
    assert a.dtype == np.float32 and np.array_equal(a, wav.numpy())
    monkeypatch.setattr(bench, "DUMP_BYTES", 3 * 10 * 4)          # room for three of the six rows
    bench.dump_outputs(str(tmp_path / "s1"), {"wav": wav})
    bench.dump_outputs(str(tmp_path / "s2"), {"wav": wav})
    s1, s2 = np.load(tmp_path / "s1" / "wav.npy"), np.load(tmp_path / "s2" / "wav.npy")
    assert s1.shape == (3, 10) and np.array_equal(s1, s2)            # fixed sample
    rows = s1[:, 0] / 10
    assert list(rows) == sorted(set(rows)) and all(np.array_equal(s1[i], wav.numpy()[int(r)]) for i, r in enumerate(rows))


def test_reference_arm_nonzero_rank_exits_quietly():
    lines = _run(["--impl", "reference", "--workload", "tiny", "--steps", "1", "--warmup", "0", "--gpus", "2"],
                 env={"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2", "MASTER_ADDR": "127.0.0.1", "MASTER_PORT": "29533"})
    assert lines == []
