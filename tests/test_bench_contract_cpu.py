"""bench.py's CPU arm (--impl reference) runs here without a GPU: check the JSON contract of the line it prints."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_contract():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    line = json.loads(r.stdout.strip().splitlines()[-1])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "cpu_baseline", "e2e", "impl"):
        assert k in line, k
    assert line["impl"] == "reference" and line["unit"] == "Mpix/s" and line["value"] > 0
    assert line["vs_baseline"] is None and line["higher_is_better"] is True
    assert set(("value", "unit", "cores", "kind", "sample")) <= set(line["cpu_baseline"])
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in line["config"]


def test_dump_outputs_is_for_the_gpu_path(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                        "--dump-outputs", str(tmp_path / "out")], capture_output=True, text=True, timeout=120)
    assert r.returncode == 2 and "--dump-outputs" in r.stderr and not (tmp_path / "out").exists()


def test_reference_arm_nonzero_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=120, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""
