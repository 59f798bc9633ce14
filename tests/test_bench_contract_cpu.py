"""bench.py contract, CPU side: the reference arm prints ONE JSON line with the keys the driver reads."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, timeout=600, env=e, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    return lines


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    lines = _run(["--impl", "reference", "--workload", "c1", "--steps", "1", "--warmup", "1"])
    assert len(lines) == 1
    j = json.loads(lines[0])
    assert j["impl"] == "reference" and j["metric"] == "index-build vectors/sec" and j["unit"] == "vectors/s"
    for key in ("value", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in j, key
    assert j["value"] > 0 and j["steps"] == 1 and j["warmup"] == 1 and j["higher_is_better"] is True
    assert j["cpu_baseline"]["kind"] == "port" and j["cpu_baseline"]["cores"] == 1        # configs[0]: single-thread CPU reference
    assert j["e2e"]["value"] == j["value"] and j["e2e"]["h2d_bytes_per_step"] == 0 and j["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in j["config"]


def test_bad_step_counts_and_dump_of_the_reference_arm_are_refused():
    for args in (["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "out"]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "c1"] + args, capture_output=True, text=True, timeout=60, cwd=ROOT)
        assert out.returncode == 2 and "error:" in out.stderr, args


def test_reference_arm_only_runs_on_rank_zero():
    assert _run(["--impl", "reference", "--workload", "c1", "--steps", "1", "--warmup", "1"], env={"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}) == []
