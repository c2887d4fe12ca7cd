"""bench.py contract on CPU: the reference arm (`--impl reference`, the CPU oracle port) prints ONE JSON line with the keys
the driver reads, on a config small enough for the CPU suite; and the committed ncu traffic table parses."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    env = dict(os.environ, LT_BENCH_CPU_THREADS="4")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                        "--layers", "18", "--image", "64", "--volume", "32", "--views", "2"],
                       capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip().startswith("{")]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "samples/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["gpu_launches"] == 0
    assert d["steps"] == 2                                    # --steps is the number of timed forwards
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] == 4 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["vs_baseline"] is None and d["scaling"] == "weak"


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                       capture_output=True, text=True, timeout=300, env=env, cwd=ROOT)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_rejects_zero_steps_and_dump_outside_the_native_arm(tmp_path):
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path / "out")]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True, timeout=300, cwd=ROOT)
        assert r.returncode == 2 and "error:" in r.stderr and r.stdout.strip() == ""
    assert not (tmp_path / "out").exists()


def test_ncu_traffic_table():
    t = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
    for k in ("conv_tc_kernel", "conv_fold_kernel", "unproject", "softargmax"):
        assert t[k] > 1e6
