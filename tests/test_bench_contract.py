"""bench.py contract checks that need no GPU: the reference arm (`--impl reference`) must print
exactly one JSON line with the keys its readers use and write the feature tables of its last timed
step with --dump-outputs, and non-zero ranks of a torchrun launch must stay silent."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(extra_env=None, extra_args=()):
    env = dict(os.environ)
    env.update(extra_env or {})
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference",
                          "--steps", "1", "--warmup", "1", *extra_args], cwd=ROOT, env=env,
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    return [l for l in out.stdout.splitlines() if l.strip()]


def test_reference_arm_prints_one_json_line():
    lines = _run()
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "klt_features_per_s"
    assert d["unit"] == "features/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["n_gpus"] == 1 and d["steps"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["e2e"]["value"] == d["value"]
    assert d["config"]["workload"].startswith("c3")
    assert d["ba"]["value"] > 0


def test_reference_arm_is_silent_on_other_ranks():
    assert _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}) == []


def test_dump_outputs_writes_the_feature_tables(tmp_path):
    assert len(_run(extra_args=["--dump-outputs", str(tmp_path)])) == 1
    shapes = {"klt_status": (4, 2000), "klt_pos": (4, 2000, 2), "klt_gain": (4, 2000), "klt_fed": (4, 2000),
              "klt_counts": (4,)}
    assert sorted(p.name for p in tmp_path.iterdir()) == sorted(n + ".npy" for n in shapes)
    for name, shape in shapes.items():
        a = np.load(tmp_path / (name + ".npy"))
        assert a.dtype == np.float32 and a.shape == shape, name
    status = np.load(tmp_path / "klt_status.npy")
    assert set(np.unique(status)) <= {-1.0, 0.0, 1.0} and (status == 0).mean() > 0.5
