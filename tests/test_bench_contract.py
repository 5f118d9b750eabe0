"""bench.py contract, the part that runs without a GPU: `--impl reference` (the CPU arm the driver
runs beside ours) prints exactly ONE JSON line on stdout with the agreed keys."""
import json
import os
import subprocess
import sys

from helpers import ROOT

REQUIRED = {"impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step",
            "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"}


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    env = dict(os.environ, OMP_NUM_THREADS="4")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                        "--warmup", "3"], capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, "stdout must carry the JSON line and nothing else"
    d = json.loads(lines[0])
    assert REQUIRED <= set(d), REQUIRED - set(d)
    assert d["impl"] == "reference" and d["metric"] == "spectrogram frames/sec" and d["unit"] == "frames/s"
    assert d["higher_is_better"] is True and d["vs_baseline"] is None and d["warmup"] >= 3
    assert d["value"] > 0 and d["n_gpus"] == 1 and d["data"] == "synthetic"
    assert d["config"]["workload"].startswith("cfg2")
    cb = d["cpu_baseline"]
    # "reference" when oracle/_ref (the unmodified reference, oracle/install_ref.sh) is installed,
    # else the NumPy oracle port
    want = "reference" if os.path.isdir(os.path.join(ROOT, "oracle", "_ref", "nnAudio")) else "port"
    assert cb["kind"] == want and cb["value"] == d["value"] and cb["cores"] >= 1 and cb["sample"]
    e2e = d["e2e"]
    assert e2e["value"] == d["value"] and e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0
