"""bench.py's reference arm (`--impl reference`: the CPU port of the hot path, the one leg of the bench that may execute oracle/)
runs without a GPU and prints ONE JSON line with the contract's keys."""
import json
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, cwd=str(ROOT))
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "ace_train_iters_per_s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["n_gpus"] == 1 and d["steps"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "iters/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0 and d["config"]["global_batch"] == 5120


def test_reference_arm_other_ranks_exit_quietly():
    import os
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=120, cwd=str(ROOT), env=env)
    assert out.returncode == 0 and not [l for l in out.stdout.splitlines() if l.startswith("{")]


def test_dump_outputs_writes_float_arrays(tmp_path):
    """`--dump-outputs DIR`: one DIR/<name>.npy per output, integer and half results widened to float64 / float32."""
    import numpy as np
    import torch
    sys.path.insert(0, str(ROOT))
    import bench
    src = {"idx": torch.arange(5, dtype=torch.int32), "h": torch.linspace(0, 1, 7).half(), "d": torch.ones(2, 3, dtype=torch.float64)}
    bench.dump_outputs(str(tmp_path / "out"), src)
    got = {p.stem: np.load(p) for p in (tmp_path / "out").glob("*.npy")}
    assert {k: v.dtype for k, v in got.items()} == {"idx": np.float64, "h": np.float32, "d": np.float64}
    for k, t in src.items():
        np.testing.assert_array_equal(got[k], t.double().numpy())
