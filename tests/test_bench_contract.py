"""What `bench.py` promises its callers, checked on a yeast-scale workload.  `--impl reference` (the CPU arm: the reference's
algorithm on the host cores): one JSON line with the agreed keys from rank 0, nothing and exit code 0 from the other ranks.
Our arm: the outputs `--dump-outputs` writes."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(env_extra):
    env = dict(os.environ, **env_extra)
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "T", "--steps", "2",
                           "--warmup", "1", "--cpu-budget-s", "5"], capture_output=True, text=True, env=env, cwd=ROOT, timeout=600)


def test_reference_arm_prints_the_contract_line():
    r = _run({})
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["unit"] == "proposals/s"
    assert d["metric"].startswith("delta-log-L proposals scored per second")
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["steps"] >= 1 and d["gpu_launches"] == 0
    assert d["config"]["workload"] == "T" and d["config"]["nnz"] == 231308 and d["config"]["n_frags"] == 900
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["vs_baseline"] is None and d["data"] == "synthetic"


def test_reference_arm_other_ranks_exit_quietly():
    r = _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r.returncode == 0 and r.stdout.strip() == ""


@pytest.mark.gpu
def test_dump_outputs_of_the_timed_path_repeat_exactly(built, tmp_path):
    """--dump-outputs: float64 arrays of the replica pass's last step, at most 64 MB, the same from run to run; --steps K
    runs K timed steps per chain"""
    steps, chains = 12, 3
    dumps = []
    for run in range(2):
        d = tmp_path / ("run%d" % run)
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "T", "--steps", str(steps), "--warmup", "2",
                            "--chains", str(chains), "--no-cpu-baseline", "--no-ref-gpu", "--dump-outputs", str(d)],
                           capture_output=True, text=True, cwd=ROOT, timeout=900)
        assert r.returncode == 0, r.stderr[-3000:]
        lines = [l for l in r.stdout.splitlines() if l.strip()]
        assert len(lines) == 1, lines
        out = json.loads(lines[0])
        assert out["steps"] == steps and "%d chains x %d steps" % (chains, steps) in out["config"]["timed"]
        files = {f.stem: np.load(f) for f in sorted(d.glob("*.npy"))}
        assert sum(f.stat().st_size for f in d.glob("*.npy")) <= 64 << 20
        assert all(a.dtype == np.float64 for a in files.values())
        dumps.append(files)
    a, b = dumps
    assert sorted(a) == sorted(b)
    nf = out["config"]["n_frags"]
    assert a["scaffold_pos"].shape == (chains, nf) and a["last_step_likelihood"].shape == (chains,)
    assert np.array_equal(a["scaffold_fragment_index"], np.arange(nf))
    for k in a:
        assert np.array_equal(a[k], b[k]), k
