"""bench.py's JSON contract: the committed round-1 line (profiles/r01_bench_line.json, produced on a B200 by
`python bench.py --steps 10 --warmup 3`) and a live run of the CPU reference arm."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches"}


def test_committed_bench_line_has_the_contract_keys():
    d = json.load(open(os.path.join(ROOT, "profiles", "r01_bench_line.json")))
    assert BASE_KEYS <= set(d)
    assert d["unit"] == "records/s" and d["higher_is_better"] is True and d["scaling"] == "weak" and d["vs_baseline"] is None
    assert d["dtype"] == "f64" and d["data"] == "synthetic" and "workload" in d["config"] and "l2" in d["config"]
    assert d["warmup"] >= 3 and d["gpu_launches"] > 0
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(d["e2e"])
    assert d["e2e"]["h2d_bytes_per_step"] == 29 * d["config"]["rows_per_gpu"] and d["e2e"]["value"] < d["value"]
    r = d["roofline"]
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    assert r["traffic"] is None or r["traffic"] > 0
    c = d["cpu_baseline"]
    assert c["kind"] == "port" and c["cores"] >= 1 and c["value"] > 0 and c["sample"]
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(d["clocks"])
    assert not set(d["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}


def test_reference_arm_runs_on_cpu():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                          "--ref-series", "2000"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads(out.stdout.strip().splitlines()[-1])
    assert d["impl"] == "reference" and BASE_KEYS <= set(d)
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] == d["value"]
    py = d["cpu_baseline"]["python_port_1core"]          # single-core pure-Python restatement, reported beside the C port
    assert py["cores"] == 1 and 0 < py["value"] < d["value"] * 50
    # ranks other than 0 print nothing and exit 0
    env = dict(os.environ, RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                          "--ref-series", "100"], capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def _dumped(out_dir):
    import numpy as np
    return {f[:-4]: np.load(os.path.join(out_dir, f)) for f in os.listdir(out_dir)}


def _oracle_rows_of_bench_table(series, points):
    sys.path.insert(0, ROOT)
    import bench
    from tests.util import oracle_rows
    return oracle_rows(bench.bench_table_numpy(series, points), "EWMA")[0]


def test_reference_arm_dumps_its_outputs(tmp_path):
    from tests.util import EXACT_COLS, SCORE_COLS, assert_same_rows
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                          "--series", "300", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads(out.stdout.strip().splitlines()[-1])
    got = _dumped(tmp_path)
    assert set(got) == set(EXACT_COLS + SCORE_COLS) and all(v.dtype.name == "float64" for v in got.values())
    assert d["outputs"]["rows"] == d["outputs"]["result_rows"] == len(got["flow_end"]) > 0
    assert_same_rows(got, _oracle_rows_of_bench_table(300, 100), what="dumped reference outputs")


@pytest.mark.gpu
def test_gpu_arm_times_steps_jobs_and_dumps_the_last_one(tmp_path):
    """--steps K times K jobs; --dump-outputs writes the rows the last of them returned, which are the oracle's."""
    from tests.util import assert_same_rows
    lines = {}
    for k in (1, 3):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--series", "3000", "--steps", str(k), "--warmup", "1",
                              "--no-cpu", "--no-sides", "--no-pipelined", "--no-parity", "--dump-outputs", str(tmp_path / str(k))],
                             capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        lines[k] = json.loads(out.stdout.strip().splitlines()[-1])
    assert lines[1]["steps"] == 1 and lines[3]["steps"] == 3
    assert lines[3]["gpu_launches"] == 3 * lines[1]["gpu_launches"] > 0
    want = _oracle_rows_of_bench_table(3000, 100)
    for k in (1, 3):
        o = lines[k]["outputs"]
        assert o["rows"] == o["result_rows"] == lines[k]["result_rows"]
        assert_same_rows(_dumped(tmp_path / str(k)), want, what="dumped outputs, --steps %d" % k)


def test_sample_mask_is_the_same_subset_for_torch_and_numpy_columns():
    """bench.py's parity key selects connections by a hash of (sourceIP, destinationIP): the device-side selection of
    input rows (torch, signed bit patterns) and the host-side selection of result rows (numpy) must agree."""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    rng = np.random.default_rng(0)
    a = rng.integers(0, 1 << 32, 20000, dtype=np.uint64).astype(np.uint32)
    b = rng.integers(0, 1 << 32, 20000, dtype=np.uint64).astype(np.uint32)
    ta = torch.from_numpy(a.view(np.int32).copy())
    tb = torch.from_numpy(b.view(np.int32).copy())
    for frac in (0.001, 0.05, 1.0):
        m_np = bench.sample_mask(a, b, frac)
        m_t = bench.sample_mask(ta, tb, frac).numpy()
        assert np.array_equal(m_np, m_t)
        assert abs(m_np.mean() - frac) < 0.01 + 0.2 * frac


def test_sharded_generator_is_balanced_and_spreads_every_connection():
    import numpy as np
    from theia_b200 import synth
    for world in (2, 4, 8):
        parts = [synth.torch_cols_to_numpy(synth.make_flows_torch_sharded(25, 100, 3, "cpu", r, world)) for r in range(world)]
        assert len({len(p["value"]) for p in parts}) == 1            # every rank holds the same number of rows
        t = {k: np.concatenate([p[k] for p in parts]) for k in parts[0]}
        key = t["src_ip"].astype(np.uint64) << np.uint64(32) | t["flow_start"].astype(np.uint64)
        _, counts = np.unique(key, return_counts=True)
        assert len(counts) == 25 * world and (counts == 100).all()
        for p in parts:                                                # a connection's points live on every rank
            k = p["src_ip"].astype(np.uint64) << np.uint64(32) | p["flow_start"].astype(np.uint64)
            assert len(np.unique(k)) == 25 * world


def test_committed_round2_line_has_parity_sides_and_a_full_size_cpu_arm():
    """profiles/r02_bench_line.json: the default `python bench.py` on a B200 at the end of round 2."""
    d = json.load(open(os.path.join(ROOT, "profiles", "r02_bench_line.json")))
    assert BASE_KEYS <= set(d) and d["n_gpus"] == 1 and d["warmup"] >= 3 and d["gpu_launches"] > 0
    assert d["parity"]["ok"] is True and d["parity"]["checked"] >= 2500          # sampled connections, bit-exact vs the oracle
    r = d["roofline"]
    assert r["bound"] == "hbm" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and r["traffic"] > 0
    assert d["e2e"]["h2d_bytes_per_step"] == 29 * d["config"]["rows_per_gpu"] and d["e2e"]["value"] < d["value"]
    c = d["cpu_baseline"]
    assert c["kind"] == "port" and c["threads_used"] == c["cores"] > 1 and "100000000 rows" in c["sample"]
    sides = {s["algo"]: s for s in d["side"]}
    assert set(sides) == {"DBSCAN", "ARIMA"}
    assert sides["DBSCAN"]["records"] == 240_000_000 and sides["DBSCAN"]["parity"]["ok"] is True
    assert sides["ARIMA"]["parity"]["ok"] is True and sides["ARIMA"]["parity"]["flags_identical"] >= 0.99
    for s in sides.values():
        assert {"bound", "achieved", "peak", "frac"} <= set(s["roofline"])
    assert not set(d["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
