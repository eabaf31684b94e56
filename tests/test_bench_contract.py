"""bench.py's reference arm is CPU-only (the oracle port on the host cores), so its JSON contract can be checked here without a GPU:
one line, `impl: reference`, the metric / unit / config of the CUDA arm, a `cpu_baseline` describing the run and an `e2e` that repeats the value."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "small", "--steps", "1", "--warmup", "3"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.strip().splitlines() if ln.startswith("{")]
    assert len(lines) == 1, out.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "spectra/sec" and d["unit"] == "spectra/s" and d["higher_is_better"] is True
    assert d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] >= 3 and d["scaling"] == "weak" and d["data"] == "synthetic"
    assert d["config"]["workload"].startswith("small:")
    assert d["value"] > 0 and d["ms_per_step"] > 0
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["unit"] == "spectra/s" and "sample" in cb
    assert d["e2e"] == {"value": d["value"], "unit": "spectra/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_rejects_arguments_it_cannot_honour():
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "small"] + extra, capture_output=True, text=True, timeout=120,
                             cwd=ROOT)
        assert out.returncode == 2 and out.stdout == "", extra


def test_dump_outputs_writes_the_psm_table_as_float_arrays(tmp_path):
    """--dump-outputs: one float32 / float64 array per Feature field, rows past a spectrum's count zeroed, at most 64 MB, and the same seeded
    sample of spectra on every run when the table is larger."""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    from sage_b200 import api
    rng = np.random.default_rng(1)
    for n, r in ((500, 2), (100_000, 5)):
        f = np.zeros(n * r, api.FEATURE_DTYPE)
        f.view(np.uint8)[:] = rng.integers(0, 256, f.nbytes, dtype=np.uint8)
        c = rng.integers(0, r + 1, n).astype(np.uint32)
        dirs = [tmp_path / f"{n}_{k}" for k in range(2)]
        for d in dirs:
            bench.dump_outputs(str(d), f, c, r)
        names = sorted(p.name for p in dirs[0].iterdir())
        assert names == sorted([x + ".npy" for x in f.dtype.names if not x.startswith("_")] + ["counts.npy", "spectra.npy"])
        assert sum(p.stat().st_size for p in dirs[0].iterdir()) <= 64 << 20
        assert all((dirs[0] / x).read_bytes() == (dirs[1] / x).read_bytes() for x in names)
        s = np.load(dirs[0] / "spectra.npy").astype(np.int64)
        assert (len(s) == n) == (n == 500) and np.all(np.diff(s) > 0)
        assert np.array_equal(np.load(dirs[0] / "counts.npy"), c[s])
        written = np.arange(r)[None, :] < c[s][:, None]
        for x in f.dtype.names:
            if x.startswith("_"):
                continue
            a, want = np.load(dirs[0] / f"{x}.npy"), f.reshape(n, r)[s][x]
            assert a.dtype == (np.float32 if want.dtype == np.float32 else np.float64) and a.shape == (len(s), r)
            assert a[written].astype(want.dtype).tobytes() == want[written].tobytes() and np.all(a[~written] == 0), x


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--workload", "small", "--steps", "1"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == "", out.stdout + out.stderr[-1000:]
