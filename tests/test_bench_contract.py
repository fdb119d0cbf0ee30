"""bench.py's JSON-line contract, the parts that need no GPU: `--impl reference` (the reference's own CPU path on the
box's host threads) prints the same `config`, `metric` and `unit` as the repo arm would for the same flags, so that the
driver's ratio compares like with like; rank != 0 of a multi-rank launch does no work."""
import json
import os
import subprocess
import sys

from common import ROOT

sys.path.insert(0, ROOT)


def _ref_line(extra=()):
    env = dict(os.environ)
    env.pop("RANK", None)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        *extra], capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


def test_reference_arm_prints_the_repo_arms_config():
    import bench
    line = _ref_line()
    assert line["impl"] == "reference" and line["higher_is_better"] is True
    curve, kind, metric, unit = bench.WORKLOADS["secp256r1_fixed_base"]
    assert (line["metric"], line["unit"]) == (metric, unit)
    # what Ours / main() put into the line for the default flags on one GPU
    want = bench.line_config("secp256r1_fixed_base", 20, 1, bench.DEFAULT_COMB[curve], bench.resolve_gather(kind, 1, "peer-root"))
    assert line["config"] == want
    assert line["e2e"] == {"value": line["value"], "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = line["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == line["value"]
    # the host description says how many CPUs' worth of time the threads really had (cgroup quota)
    assert 1 <= cb["host"]["effective_cpus"] <= cb["host"]["affinity_cpus"]


def test_reference_arm_config_at_eight_ranks_names_the_gather():
    import bench
    line = _ref_line(["--gpus", "8"])
    want = bench.line_config("secp256r1_fixed_base", 20, 8, bench.DEFAULT_COMB["SECP256R1"], "peer-root")
    assert line["config"] == want and line["config"]["global_batch"] == 8 << 20 and line["n_gpus"] == 8


def test_other_ranks_of_the_reference_arm_exit_without_work():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                        "--warmup", "0"], capture_output=True, text=True, timeout=300, env=env, cwd=ROOT)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_reference_arm_dumps_the_last_steps_outputs(tmp_path):
    """--dump-outputs: float32 / float64 .npy files under 64 MB, identical for two runs with the same arguments."""
    import numpy as np
    runs = []
    for name in ("a", "b"):
        _ref_line(["--batch-log2", "8", "--dump-outputs", str(tmp_path / name)])
        files = sorted(os.listdir(tmp_path / name))
        assert files == ["points.npy", "sample_index.npy", "status.npy"]
        runs.append({f[:-4]: np.load(tmp_path / name / f) for f in files})
    a, b = runs
    assert sum(x.nbytes for x in a.values()) <= 64 << 20
    assert all(x.dtype in (np.float32, np.float64) for x in a.values())
    assert a["points"].shape == (256, 64) and a["status"].shape == (256,)
    assert set(np.unique(a["status"])) <= {0.0, 1.0}
    assert all((a[f] == b[f]).all() for f in a)
