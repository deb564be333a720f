"""bench.py's reference arm runs on the host alone, so its JSON contract can be checked without a GPU."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line(oracle_mod):
    pr = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                         "--ref-pairs", "96"], capture_output=True, text=True, timeout=600)
    assert pr.returncode == 0, pr.stderr[-500:]
    lines = [ln for ln in pr.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "GCUPS" and d["higher_is_better"] is True
    for key in ("metric", "value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data", "config",
                "cpu_baseline", "e2e", "gpu_launches"):
        assert key in d, key
    assert d["value"] > 0 and d["gpu_launches"] == 0
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]
    assert "workload" in d["config"]


def test_reference_arm_other_ranks_exit_quietly(oracle_mod):
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    pr = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                        capture_output=True, text=True, timeout=120, env=env)
    assert pr.returncode == 0 and pr.stdout.strip() == ""


def test_steps_below_one_is_refused():
    pr = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True, timeout=120)
    assert pr.returncode == 2 and "--steps must be at least 1" in pr.stderr and pr.stdout == ""


def _bench_module():
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _synthetic_result(n, seed=1):
    import numpy as np
    from aligntools.c_b200 import BatchResult
    rng = np.random.default_rng(seed)
    r = BatchResult(n)
    for k in ("score", "end_i", "end_j", "beg_i", "beg_j"):
        getattr(r, k)[:] = rng.integers(0, 500, n)
    r.cigar_off = np.zeros(n + 1, np.uint64)
    np.cumsum(rng.integers(0, 12, n), out=r.cigar_off[1:])
    r.cigar = rng.integers(0, 1 << 14, int(r.cigar_off[-1]) + 1).astype(np.uint32)
    return r


def _load_dump(d):
    import numpy as np
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def _check_dump(r, got):
    import numpy as np
    idx = got["pair_index"].astype(np.int64) if "pair_index" in got else np.arange(r.n)
    off = got["cigar_off"].astype(np.int64)
    assert got["cigar_off"].dtype == np.float64 and len(off) == len(idx) + 1 and off[0] == 0
    for k in ("score", "end_i", "end_j", "beg_i", "beg_j"):
        assert got[k].dtype == np.float32 and np.array_equal(got[k], getattr(r, k)[idx]), k
    assert got["cigar"].dtype == np.float32 and len(got["cigar"]) == off[-1]
    for x, p in enumerate(idx):
        assert np.array_equal(got["cigar"][off[x]:off[x + 1]], r.cigar_ops(p)), p
    return idx


def test_dump_outputs_whole_result(tmp_path):
    bench = _bench_module()
    r = _synthetic_result(3000)
    bench.dump_outputs(r, str(tmp_path / "d"))
    got = _load_dump(tmp_path / "d")
    assert "pair_index" not in got
    _check_dump(r, got)


def test_dump_outputs_seeded_sample_within_budget(tmp_path, monkeypatch):
    """A result larger than the budget is cut to a seeded sample of whole pairs that fits it, the same on every run."""
    import numpy as np
    bench = _bench_module()
    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", 64 << 10)
    r = _synthetic_result(3000)
    for d in ("a", "b"):
        bench.dump_outputs(r, str(tmp_path / d))
        assert sum(os.path.getsize(tmp_path / d / f) for f in os.listdir(tmp_path / d)) <= 64 << 10
    a, b = _load_dump(tmp_path / "a"), _load_dump(tmp_path / "b")
    assert a.keys() == b.keys() and all(np.array_equal(a[k], b[k]) for k in a)
    idx = _check_dump(r, a)
    assert 0 < len(idx) < r.n and np.all(np.diff(idx) > 0)
