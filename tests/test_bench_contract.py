"""bench.py contract, as far as it can be checked without a GPU: the reference arm prints ONE JSON line with the agreed
keys (and uses all host cores even when the launcher exports OMP_NUM_THREADS=1, as torch.distributed.run does), and our
arm refuses to run without a CUDA device instead of falling back to anything."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(args, env_extra=None):
    env = dict(os.environ)
    env.update(env_extra or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, timeout=600, env=env)


def test_reference_arm_line():
    r = run_bench(["--impl", "reference", "--workload", "c2", "--steps", "1", "--warmup", "1"], {"OMP_NUM_THREADS": "1"})
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert key in d, key
    assert d["impl"] == "reference" and d["unit"] == "pairs/s" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["gpu_launches"] == 0 and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["e2e"]["value"] == d["value"] == d["cpu_baseline"]["value"] > 0
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and "workload" in d["config"]
    try:
        cores = len(os.sched_getaffinity(0))
    except AttributeError:
        cores = os.cpu_count()
    assert d["cpu_baseline"]["cores"] == cores   # not the launcher's OMP_NUM_THREADS=1


def test_non_zero_ranks_of_the_reference_arm_stay_silent():
    r = run_bench(["--impl", "reference", "--workload", "c2", "--steps", "1", "--warmup", "1", "--gpus", "2"],
                  {"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_our_arm_needs_a_gpu():
    r = run_bench(["--workload", "c2", "--steps", "1"], {"CUDA_VISIBLE_DEVICES": ""})   # any device hidden from the run
    assert r.returncode != 0 and r.stdout.strip() == "" and "no CUDA device" in r.stderr
