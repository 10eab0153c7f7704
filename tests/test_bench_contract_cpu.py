"""bench.py's reference arm runs on the host cores alone (oracle/c, C++/OpenMP): its JSON line is checked here against the
driver's contract on a small grid (the GPU arm prints the same keys; it needs a B200).  The GPU arm's --dump-outputs writer is
checked on host arrays."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--grid", "256", "--steps", "2", "--warmup", "3",
                        "--ref-batches", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1                                   # ONE JSON line
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "impl", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "steps/s" and d["higher_is_better"] is True and d["dtype"] == "f64"
    assert d["steps"] == 2 and d["warmup"] == 3 and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert "workload" in d["config"] and "model" not in d["config"] and d["config"]["grid"] == [256, 256]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["value"] == d["value"] and cb["cores"] >= 1 and "sample" in cb
    assert d["e2e"] == {"value": d["value"], "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["details"]["sample_steps"] == 10 and d["value"] > 0
    hr = cb["host_roofline"]
    assert hr["unit"] == "GB/s" and hr["achieved"] > 0 and hr["peak"] > 0 and hr["blas1_gbytes"] > hr["spmv_gbytes"] > 0


def test_reference_arm_other_ranks_exit_without_work():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--grid", "256"],
                       capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_dump_outputs_writes_float64_arrays_and_a_fixed_sample_of_long_vectors(tmp_path):
    import types
    import numpy as np
    import bench
    n = bench.DUMP_MAX_ENTRIES + 5
    rng = np.random.default_rng(3)
    st = types.SimpleNamespace(z_u=rng.standard_normal(n), z_p=-0.2, tau_u=rng.standard_normal(n), tau_p=0.1)
    rows = [dict(param=-0.1 - 1e-3 * k, x=1.0 + k, itnewton=2, itlinear=30 + k, ds=-1e-3, step=k, n_unstable=-1) for k in range(3)]
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), rows, st)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == ["branch.npy", "p.npy", "tau_p.npy", "tau_u.npy", "u.npy"]
    for f in names:
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype == np.float64 and np.array_equal(a, b)           # the same entries on every run
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in names) <= 64 << 20
    u, tau = np.load(tmp_path / "a" / "u.npy"), np.load(tmp_path / "a" / "tau_u.npy")
    assert u.shape == tau.shape == (bench.DUMP_MAX_ENTRIES,)
    idx = np.searchsorted(np.sort(st.z_u), u)                           # a sample of the state, in index order
    assert np.array_equal(np.sort(st.z_u)[idx], u)
    pos = np.argsort(st.z_u)[idx]
    assert np.all(np.diff(pos) > 0) and np.array_equal(st.tau_u[pos], tau)
    assert np.load(tmp_path / "a" / "branch.npy").tolist()[2] == [-0.1 - 2e-3, 3.0, 2.0, 32.0, -1e-3, 2.0, -1.0]
    assert np.load(tmp_path / "a" / "p.npy").tolist() == [-0.2] and np.load(tmp_path / "a" / "tau_p.npy").tolist() == [0.1]
