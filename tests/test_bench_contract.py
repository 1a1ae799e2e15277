"""bench.py contract on a CPU-only box: the reference arm (`--impl reference`) runs the oracle on the host cores and
prints ONE JSON line with the agreed keys; ranks other than 0 print nothing and exit 0."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(env_extra):
    env = dict(os.environ)
    env.update(env_extra)
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", "c1", "--steps", "1", "--warmup", "1"],
                          capture_output=True, text=True, env=env, timeout=600, cwd=ROOT)


def test_reference_arm_json_line():
    p = _run({"RANK": "0", "WORLD_SIZE": "1"})
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["value"] > 0 and d["higher_is_better"] is True
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"]


def test_reference_arm_other_ranks_are_silent():
    p = _run({"RANK": "1", "WORLD_SIZE": "2"})
    assert p.returncode == 0 and p.stdout.strip() == ""


def test_dump_outputs_dtypes_budget_and_fixed_sample(tmp_path):
    """bench.py --dump-outputs: float64 stays float64, other floating types become float32, small arrays are written
    whole, and an array over what is left of the byte budget keeps the same seeded sample of rows on every call."""
    import numpy as np
    import torch

    import bench

    g = torch.Generator().manual_seed(1)
    outs = {"forces": torch.randn(50, 3, generator=g, dtype=torch.float64), "total_energy": torch.randn(1, 1, generator=g, dtype=torch.float64),
            "edge_features": torch.randn(4000, 16, generator=g).to(torch.bfloat16)}
    budget = 60_000
    for d in ("a", "b"):
        bench.dump_outputs(outs, str(tmp_path / d), budget=budget)
    got = {p.stem: np.load(p) for p in (tmp_path / "a").iterdir()}
    assert sorted(got) == sorted(outs)
    assert got["forces"].dtype == np.float64 and np.array_equal(got["forces"], outs["forces"].numpy())
    assert got["total_energy"].shape == (1, 1)
    ef = got["edge_features"]
    small = outs["forces"].numel() * 8 + 8
    assert ef.dtype == np.float32 and ef.shape == ((budget - small) // (16 * 4), 16)  # the bytes the small arrays leave
    assert sum(a.nbytes for a in got.values()) <= budget
    full = outs["edge_features"].float().numpy()
    rows = [int(np.flatnonzero((full == r).all(1))[0]) for r in ef]
    assert rows == sorted(rows) and len(set(rows)) == len(rows)  # distinct rows of the output, in ascending order
    assert np.array_equal(ef, np.load(tmp_path / "b" / "edge_features.npy"))
