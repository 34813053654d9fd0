"""bench.py keeps the driver's JSON contract (reference arm runs on CPU; tiny sample here)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    env = dict(os.environ, FB_BENCH_REF_ROWS="20000")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
                        "--warmup", "1"], capture_output=True, text=True, timeout=300, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.strip().splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
              "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "rows/s" and d["steps"] == 2 and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] == 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"]


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, FB_BENCH_REF_ROWS="20000", RANK="1", WORLD_SIZE="2")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                       capture_output=True, text=True, timeout=300, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_steps_below_one_is_an_error():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 2 and "--steps" in r.stderr and r.stdout.strip() == ""


def test_dump_outputs_writes_a_seeded_exact_float64_sample(tmp_path):
    import numpy as np

    script = f"""
import sys, types
import numpy as np, torch
sys.path.insert(0, {ROOT!r})
import bench
from fugue_b200.table import B200Table

rng = np.random.default_rng(1)
n = 1000
cols = [torch.from_numpy(rng.integers(-2**63, 2**63 - 1, n, dtype=np.int64)), torch.from_numpy(rng.standard_normal(n))]
t = B200Table("k:long,v:double", cols, offsets=torch.tensor([0, 400, 1000], dtype=torch.int64))
bench.DUMP_ROWS = 64
for d in ("a", "b"):
    bench.dump_outputs(types.SimpleNamespace(native=t), sys.argv[1] + "/" + d)
np.save(sys.argv[1] + "/k.npy", cols[0].numpy())
np.save(sys.argv[1] + "/v.npy", cols[1].numpy())
"""
    r = subprocess.run([sys.executable, "-c", script, str(tmp_path)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    a, b = tmp_path / "a", tmp_path / "b"
    names = sorted(p.name for p in a.iterdir())
    assert names == ["k_hi32.npy", "k_lo32.npy", "offsets.npy", "row_index.npy", "v.npy"]
    got = {p[:-4]: np.load(a / p) for p in names}
    for name in names:
        assert got[name[:-4]].dtype == np.float64 and np.array_equal(got[name[:-4]], np.load(b / name)), name
    rows = got["row_index"].astype(np.int64)
    assert len(rows) == 64 and np.all(np.diff(rows) > 0) and rows[-1] < 1000
    k = got["k_hi32"].astype(np.int64) * 2**32 + got["k_lo32"].astype(np.int64)
    assert np.array_equal(k, np.load(tmp_path / "k.npy")[rows])
    assert np.array_equal(got["v"], np.load(tmp_path / "v.npy")[rows])
    assert np.array_equal(got["offsets"], [0, 400, 1000])
