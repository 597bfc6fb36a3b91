"""CPU: the reference arm of bench.py honours the driver's contract (one JSON line, the agreed keys)."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "msm_mpts_per_s" and d["unit"] == "Mpts/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["steps"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": "Mpts/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]
    # --dump-outputs: the commitments of the timed step, exact as 32-bit limbs in float64
    from oracle import oracle as O
    assert sorted(os.listdir(tmp_path)) == ["commitments.npy"]
    got = np.load(tmp_path / "commitments.npy")
    assert got.dtype == np.float64 and got.shape == (d["config"]["sampled_cols_per_step"], 2, 8)
    limbs = got.astype(np.uint32).view(np.uint64).reshape(-1, 8)
    n = 1 << d["config"]["k"]
    assert (limbs[0] == O.best_multiexp_affine(O.fr_fill(n, 7000), O.gen_bases(n))).all()


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""
