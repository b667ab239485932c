"""bench.py contract checks: the reference arm prints ONE JSON line with the agreed keys (no GPU needed); on a GPU, --steps sets
the timed window and --dump-outputs writes what its last step computed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "rows/s" and d["higher_is_better"] is True
    assert d["metric"] == "RealNVP fit rows/sec (fwd+bwd+Adam)" and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload"].startswith("c3")


def test_flops_per_row_matches_the_survey_table():
    sys.path.insert(0, ROOT)
    from bench import flops_per_row, WORKLOADS
    want = {"c2": (960, 2520), "c3": (327680, 909312), "c4": (983040, 2736128), "c5": (2621440, 7208960)}   # SURVEY.md 8d
    for name, (fwd, fit) in want.items():
        D, Cd, L, hidden, _, _ = WORKLOADS[name]
        assert flops_per_row(D, Cd, L, hidden[0]) == (fwd, fit), name


@pytest.mark.gpu
def test_steps_and_dump_outputs(tmp_path):
    runs = {}
    for k in (2, 3):
        out = tmp_path / f"steps{k}"
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(k), "--warmup", "3", "--no-e2e",
                            "--no-sustained", "--no-others", "--no-cpu-baseline", "--dump-outputs", str(out)],
                           capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-2000:]
        lines = [l for l in r.stdout.splitlines() if l.strip()]
        assert len(lines) == 1, lines
        d = json.loads(lines[0])
        assert d["steps"] == k
        arrays = {f.stem: np.load(f) for f in out.iterdir()}
        assert set(arrays) == {"loss", "params", "adam_exp_avg", "adam_exp_avg_sq"}
        assert all(a.dtype == np.float32 and np.isfinite(a).all() for a in arrays.values())
        assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
        assert float(arrays["loss"]) == d["config"]["final_loss"]
        runs[k] = d, arrays
    # the timed window holds exactly --steps steps, and the dumped weights are those after the last of them
    assert runs[3][0]["gpu_launches"] * 2 == runs[2][0]["gpu_launches"] * 3
    assert not np.array_equal(runs[2][1]["params"], runs[3][1]["params"])
