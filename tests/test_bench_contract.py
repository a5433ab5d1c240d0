"""bench.py contract checks, all but the last --dump-outputs one without a GPU: the reference arm prints one JSON line with
the keys the driver reads (it runs the reference's own CPU program -- oracle/_ref -- or the oracle port)."""
import json
import os
import subprocess
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parents[1]


@pytest.mark.timeout(600)
def test_reference_arm_json_line(oracle):
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=580, cwd=str(ROOT))
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "attention_tflops" and d["unit"] == "TFLOP/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1
    assert d["value"] > 0 and d["e2e"]["value"] == d["value"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and "rows" in cb["sample"]
    assert d["config"]["m"] == 8192 and d["config"]["n"] == 65536


def test_our_arm_refuses_without_gpu(sdpa):
    """Every device is hidden from the child, so this runs the same on a GPU machine."""
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--steps", "1"], capture_output=True, text=True, timeout=300, cwd=str(ROOT),
                       env={**os.environ, "CUDA_VISIBLE_DEVICES": ""})
    assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)


def test_clock_sampler_summary_and_graceful_start():
    """bench.py's clock sampler: idle samples are dropped, the median / reasons / power come from the loaded ones;
    without NVML or nvidia-smi (this container) start() returns an inert sampler instead of failing."""
    sys.path.insert(0, str(ROOT))
    import bench
    s = bench.ClockSampler(0, None, allow_subprocess=False)
    s.rows = [(1965.0, 1965.0, 120.0, []), (1800.0, 1965.0, 900.0, ["sw_power_cap"]), (1780.0, 1965.0, 950.0, ["sw_power_cap"]),
              (1770.0, 1965.0, 910.0, [])]
    out = s.summary()
    assert out["sm_mhz"] == 1780.0 and out["sm_max_mhz"] == 1965.0 and out["samples"] == 3
    assert out["reasons"] == ["sw_power_cap"] and out["power_w_max"] == 950.0
    live = bench.ClockSampler(0, None, allow_subprocess=False).start()
    with live:
        pass
    live.close()
    assert live.summary()["samples"] >= 0


def test_steps_must_be_positive():
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--steps", "0"], capture_output=True, text=True, timeout=300, cwd=str(ROOT))
    assert r.returncode == 2 and "--steps must be at least 1" in r.stderr


def test_dump_outputs_writes_the_result_or_a_seeded_row_sample(tmp_path, monkeypatch):
    sys.path.insert(0, str(ROOT))
    import numpy as np
    import bench
    res = np.random.default_rng(0).standard_normal((300, 128))
    bench.dump_outputs(str(tmp_path / "all"), res)
    assert sorted(p.name for p in (tmp_path / "all").iterdir()) == ["result.npy"]
    assert np.array_equal(np.load(tmp_path / "all" / "result.npy"), res)
    monkeypatch.setattr(bench, "DUMP_BYTES_MAX", 100 * 128 * 8)       # room for fewer than 100 of the 300 rows
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), res)
    got, rows = np.load(tmp_path / "a" / "result.npy"), np.load(tmp_path / "a" / "result_rows.npy")
    assert got.dtype == np.float64 and rows.dtype == np.float64
    assert got.nbytes + rows.nbytes <= bench.DUMP_BYTES_MAX and 0 < len(rows) < 100
    assert np.all(np.diff(rows) > 0) and np.array_equal(got, res[rows.astype(np.int64)])
    assert np.array_equal(rows, np.load(tmp_path / "b" / "result_rows.npy"))      # the same sample every run


@pytest.mark.gpu
@pytest.mark.timeout(900)
def test_dump_outputs_is_the_timed_result(oracle, tmp_path):
    """--dump-outputs writes what the last timed step returned: the full [m, dv] fp64 result, within the bf16 path's tolerance
    of the fp64 oracle on the parity rows.  --steps sets the passes the timed region runs: with stage marks on every pass, the
    library's count of marked passes between the two reads around the timed loop is --steps."""
    import numpy as np
    sys.path.insert(0, str(ROOT))
    import bench
    m, n = 512, 4096
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--gpus", "1", "--steps", "3", "--warmup", "1", "--m", str(m),
                        "--n-per-gpu", str(n), "--extra", "none", "--no-alone", "--no-cpu-baseline", "--stage-timing-every", "1",
                        "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=880, cwd=str(ROOT))
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert line["steps"] == 3 and line["stage_ms_per_step"]["passes_timed"] == 3
    assert line["config"]["m"] == m and line["config"]["n"] == n
    assert sorted(p.name for p in tmp_path.iterdir()) == ["result.npy"]
    got = np.load(tmp_path / "result.npy")
    assert got.shape == (m, bench.DV) and got.dtype == np.float64
    rows = bench.parity_rows(m)
    np.testing.assert_allclose(got[rows], bench.oracle_rows(m, [n], rows), rtol=0, atol=bench.CONFIGS["c3"]["tol"])


def test_bench_config_shapes_match_baseline():
    """c2/c4/c5 are run at the shapes BASELINE.json states; c3 keeps 65536 keys per GPU (weak scaling)."""
    sys.path.insert(0, str(ROOT))
    import bench
    assert bench.config_shape("c3", 8) == (8192, [65536] * 8)
    assert bench.config_shape("c2", 1) == (4096, [4096])
    assert bench.config_shape("c4", 4) == (16384, [65536] * 4)
    assert bench.config_shape("c5", 8) == (32768, [131072] * 8)
    m, rows = bench.config_shape("c5", 3)          # ragged owner_count split when run on another GPU count
    assert m == 32768 and sum(rows) == 1048576 and rows == [349526, 349525, 349525]
    assert bench.EXTRAS_BY_GPUS == {1: ["c2"], 4: ["c4"], 8: ["c5"]}


def test_bench_parity_inputs_are_reproducible(oracle):
    """The oracle check in bench.py regenerates every rank's shard from its seed on rank 0: the regenerated arrays must be
    the ones the ranks built, and the row subset must be the same on every call."""
    sys.path.insert(0, str(ROOT))
    import numpy as np
    import bench
    shard_rows = [7, 5, 0, 3]
    m = 50
    rows = bench.parity_rows(m)
    assert len(rows) == 50 and (rows == bench.parity_rows(m)).all()
    assert len(bench.parity_rows(100000)) == bench.PARITY_ROWS
    got = bench.oracle_rows(m, shard_rows, rows[:9])
    K = np.concatenate([bench.make_shard(r, c)[0].numpy() for r, c in enumerate(shard_rows)])
    V = np.concatenate([bench.make_shard(r, c)[1].numpy() for r, c in enumerate(shard_rows)])
    ref = oracle.attention_f64(bench.make_q(m).numpy()[rows[:9]], K, V)
    np.testing.assert_allclose(got, ref, rtol=0, atol=1e-13)
    a, b = bench.make_shard(3, 11), bench.make_shard(3, 11)
    assert (a[0] == b[0]).all() and (a[1] == b[1]).all()
    assert not (bench.make_shard(2, 11)[0] == a[0]).all()
