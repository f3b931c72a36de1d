"""CPU: the reference arm of bench.py (`--impl reference`) runs without a GPU -- it times the reference's own
PairPollable::Send/Recv (oracle/_ref, or the port when _ref is absent) on the host cores -- and prints one
JSON line with the keys the bench contract names."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
                          "--warmup", "1", "--conns", "8", "--msg-bytes", str(256 * 1024), "--ring-kb", "1024"],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "GB/s" and line["higher_is_better"] is True
    for k in ("metric", "value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "dtype", "data", "config",
              "cpu_baseline", "e2e"):
        assert k in line, k
    assert line["value"] > 0 and line["gpu_launches"] == 0
    assert line["steps"] == 2
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0


def test_reference_arm_on_other_ranks_exits_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, timeout=120, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""
