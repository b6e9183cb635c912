"""CPU checks of bench.py's contract: the reference arm runs end to end here (it needs no GPU) and prints
the JSON line the driver parses, with the same `config.workload` string as the GPU arm would print."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_line_and_workload_label():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "config2",
                          "--cols", "12", "--rows", "300", "--steps", "2", "--warmup", "1", "--ref-budget", "0.2"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "column-pairs/sec" and line["unit"] == "pairs/s"
    assert line["higher_is_better"] is True and line["value"] > 0 and line["steps"] == 2
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"] == {"value": line["value"], "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    sys.path.insert(0, ROOT)
    import bench
    # both arms label the workload through one function (the driver compares the strings)
    assert line["config"]["workload"] == bench.workload_label("config2", 300, 12, "global")
    assert bench.workload_label("target", 20000, 2000, "global").startswith("target: 20000 features x 2000 samples")
    # defaults the driver relies on: the target workload, strong scaling, >= 3 warm-up steps
    src = open(os.path.join(ROOT, "bench.py")).read()
    assert 'add_argument("--workload", default="target"' in src and 'add_argument("--scaling", default="strong"' in src


def test_dump_outputs_full_and_sampled(tmp_path, monkeypatch):
    """--dump-outputs: float32/float64 .npy files within the byte budget; a larger result set is written as
    the same seeded sample of pairs on every run, with the pairs' positions in pair_index."""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    P = 5000
    rng = np.random.default_rng(1)
    res = {k: rng.normal(size=P) for k in ("raw", "pvalue", "taumax", "completeness")}
    res["status"] = rng.integers(0, 5, size=P).astype(np.int32)
    res["max_taumax"] = 0.75

    def load(d):
        return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}

    bench.dump_outputs(str(tmp_path / "full"), res, P)
    full = load(tmp_path / "full")
    assert sorted(full) == ["completeness", "max_taumax", "pair_index", "pvalue", "raw", "status", "taumax"]
    assert all(v.dtype in (np.float32, np.float64) for v in full.values())
    assert np.array_equal(full["pair_index"], np.arange(P)) and full["max_taumax"].tolist() == [0.75]
    assert np.array_equal(full["raw"], res["raw"]) and np.array_equal(full["status"], res["status"])

    monkeypatch.setattr(bench, "DUMP_BYTES", 4096 + 44 * 1000)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), res, P)
    a, b = load(tmp_path / "a"), load(tmp_path / "b")
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= bench.DUMP_BYTES
    sel = a["pair_index"].astype(np.int64)
    assert sel.size == 1000 and np.all(np.diff(sel) > 0)
    for k in ("raw", "pvalue", "taumax", "completeness", "status"):
        assert np.array_equal(a[k], res[k][sel]) and np.array_equal(a[k], b[k]), k


def test_steps_must_be_positive():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert out.returncode != 0 and "--steps" in out.stderr


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="3", WORLD_SIZE="8", LOCAL_RANK="3")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "8"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""
