"""bench.py's reference arm (the CPU oracle dataflow) runs without a GPU: its JSON line is checked
against the driver's contract here, and the GPU arm is checked to refuse to run without CUDA."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(*args, env=None):
    return subprocess.run(
        [sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=600, env=env
    )


def test_reference_arm_prints_one_contract_line():
    p = run_bench("--impl", "reference", "--sf", "1", "--steps", "3", "--warmup", "3")
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1  # exactly one JSON line on stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference"
    assert d["metric"] == "update_rows_per_sec" and d["unit"] == "rows/s" and d["higher_is_better"] is True
    assert d["n_gpus"] == 1 and d["steps"] == 3 and d["warmup"] >= 3
    assert d["value"] > 0 and d["ms_per_step"] > 0
    assert d["scaling"] == "weak" and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert "workload" in d["config"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    e = d["e2e"]
    assert e["value"] == d["value"] and e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0


def test_reference_arm_other_ranks_stay_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    p = run_bench("--impl", "reference", "--gpus", "2", "--sf", "1", "--steps", "3", "--warmup", "3", env=env)
    assert p.returncode == 0, p.stderr[-2000:]
    assert p.stdout.strip() == ""


DUMP_FIELDS = ("key", "count", "sum", "flags", "time", "diff")


def load_dump(d):
    import numpy as np

    return {f: np.load(os.path.join(d, f + ".npy")) for f in DUMP_FIELDS}


def consolidated(dump):
    """The dumped rows as {(key, count, sum, flags, time): diff}, equal rows summed, zero diffs dropped."""
    acc = {}
    for r in zip(*(dump[f].tolist() for f in DUMP_FIELDS)):
        acc[r[:-1]] = acc.get(r[:-1], 0) + r[-1]
    return {k: v for k, v in acc.items() if v != 0}


def test_reference_arm_dumps_the_last_timed_step(tmp_path):
    """--dump-outputs writes one float64 array per output field, the same from run to run."""
    import numpy as np

    args = ("--impl", "reference", "--sf", "1", "--steps", "3", "--warmup", "3", "--dump-outputs")
    dumps = []
    for name in ("a", "b"):
        p = run_bench(*args, str(tmp_path / name))
        assert p.returncode == 0, p.stderr[-2000:]
        dumps.append(load_dump(tmp_path / name))
    a, b = dumps
    assert all(a[f].dtype == np.float64 and a[f].shape == a["key"].shape for f in DUMP_FIELDS)
    assert len(a["key"]) > 0 and set(a["diff"].tolist()) <= {-1.0, 1.0}
    assert len(set(a["time"].tolist())) == 1  # one timestamp: the last timed step's
    assert all(np.array_equal(a[f], b[f]) for f in DUMP_FIELDS)
    # the step before has another timestamp
    p = run_bench("--impl", "reference", "--sf", "1", "--steps", "2", "--warmup", "3", "--dump-outputs", str(tmp_path / "c"))
    assert p.returncode == 0, p.stderr[-2000:]
    assert load_dump(tmp_path / "c")["time"][0] == a["time"][0] - 1


@pytest.mark.gpu
def test_gpu_arm_dump_matches_the_oracle(tmp_path):
    """The GPU arm's dump of its last timed step holds the CPU oracle's output corrections of that step."""
    args = ("--sf", "1", "--steps", "3", "--warmup", "3", "--no-cpu-baseline", "--dump-outputs")
    p = run_bench(*args, str(tmp_path / "gpu"))
    assert p.returncode == 0, p.stderr[-2000:]
    p = run_bench("--impl", "reference", *args, str(tmp_path / "cpu"))
    assert p.returncode == 0, p.stderr[-2000:]
    gpu, cpu = consolidated(load_dump(tmp_path / "gpu")), consolidated(load_dump(tmp_path / "cpu"))
    assert len(cpu) > 0 and gpu == cpu


def test_gpu_arm_fails_loudly_without_cuda():
    """The product path has no CPU fallback: without a GPU the bench must fail, not time the oracle."""
    import torch

    if torch.cuda.is_available():
        import pytest

        pytest.skip("a GPU is present")
    p = run_bench("--steps", "3", "--warmup", "3", "--sf", "1")
    assert p.returncode != 0
    assert '"metric"' not in p.stdout
