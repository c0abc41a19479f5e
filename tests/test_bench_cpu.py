"""bench.py pieces that run without a GPU: the reference arm (C oracle on the host cores, same records as the GPU
arm, CPU per-time-step latency leg) and the sharding of the record blocks over the ranks."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--scenarios", "8",
                          "--steps", "2", "--warmup", "1", "--no-cache", "--sim-steps", "6", "--gen-workers", "1"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "vehicle-plans/sec" and line["unit"] == "plans/s"
    assert line["higher_is_better"] is True and line["steps"] == 2 and line["warmup"] == 1
    n = line["config"]["searches_per_step_per_gpu"]
    assert n == 8 * 6 * 20 and "same records in both arms" in line["config"]["workload"]
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == line["value"] and f"all {n} search records" in cb["sample"]
    lat = cb["latency_ms_per_timestep"]
    assert lat["n"] == 2 * 8 * 6 and 0 < lat["p50"] <= lat["p99"] <= lat["max"]
    assert line["e2e"] == {"value": line["value"], "unit": "plans/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert abs(line["value"] - n * 2 / (line["ms_per_step"] * 2e-3)) < 1e-6 * line["value"]


def test_rank_blocks_weak_and_strong():
    sys.path.insert(0, ROOT)
    import bench

    class A:
        scenarios, scenarios_total = 512, 0
    assert bench.rank_blocks(A, 0, 1) == list(range(64)) and bench.rank_blocks(A, 3, 8) == list(range(192, 256))
    A.scenarios_total = 4096
    parts = [bench.rank_blocks(A, r, 8) for r in range(8)]
    assert sorted(b for p in parts for b in p) == list(range(512)) and all(len(p) == 64 for p in parts)
    assert parts[1][:3] == [1, 9, 17]                                   # block-cyclic
    cfg = bench.workload_config(type("X", (), {"scenarios_total": 4096, "scenarios": 512, "sim_steps": 35, "optimizer": "graph",
                                               "vehicles": 20, "mpa": "triple_speed", "mcts_expansions": 250}), 8, 358400, 6)
    assert "4096 scenarios in total" in cfg["workload"] and cfg["searches_per_step_per_gpu"] == 358400


def test_dump_outputs_is_float_exact_bounded_and_seeded(tmp_path):
    """--dump-outputs: every field of the result as float64 (the 64-bit pop hash in two exact halves), all finite (the
    NaN plans of exhausted searches as 0); past the byte limit a sample of searches that is the same from run to run."""
    sys.path.insert(0, ROOT)
    import bench
    from pdmpc_b200.records import BatchResult
    rng = np.random.default_rng(5)
    res = BatchResult.empty(300, 6)
    res.pop_hash[:] = rng.integers(0, 2**64, 300, dtype=np.uint64)
    res.trims[:] = rng.integers(1, 13, res.trims.shape)
    res.y_predicted[:] = rng.standard_normal(res.y_predicted.shape)
    res.g_path[:] = rng.random(res.g_path.shape)
    ex = rng.random(300) < 0.2
    res.is_exhausted[ex] = 1
    res.y_predicted[ex] = res.g_path[ex] = res.h_path[ex] = np.nan

    def load(d):
        return {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d)}

    bench.dump_outputs(res, str(tmp_path / "all"), bench.DUMP_LIMIT)
    full = load(tmp_path / "all")
    assert np.array_equal(full["rows"], np.arange(300))
    assert all(np.isfinite(v).all() for v in full.values())
    assert np.array_equal(full["is_exhausted"], ex) and (full["g_path"][ex] == 0).all() and (full["y_predicted"][ex] == 0).all()
    assert np.array_equal(full["g_path"][~ex], res.g_path[~ex])
    for d in ("a", "b"):
        bench.dump_outputs(res, str(tmp_path / d), 40000)
    a, b = load(tmp_path / "a"), load(tmp_path / "b")
    assert sorted(a) == sorted(full) and all(v.dtype == np.float64 for v in a.values())
    assert sum(v.nbytes for v in a.values()) <= 40000
    rows = a["rows"].astype(np.int64)
    assert 0 < rows.size < 300 and (np.diff(rows) > 0).all()
    for k in a:
        assert np.array_equal(a[k], b[k]) and np.array_equal(a[k], full[k][rows])
    h = (a["pop_hash_hi"].astype(np.uint64) << np.uint64(32)) | a["pop_hash_lo"].astype(np.uint64)
    assert np.array_equal(h, res.pop_hash[rows])
    assert np.array_equal(a["trims"], res.trims[rows])
    assert np.array_equal(a["y_predicted"][~ex[rows]], res.y_predicted[rows][~ex[rows]])
    assert np.isnan(res.g_path[ex]).all()                                # the caller's result is left as it was
    res.h_path[np.flatnonzero(~ex)[0], 2] = np.nan                       # NaN in a plan that exists: a wrong result
    with pytest.raises(RuntimeError, match="h_path"):
        bench.dump_outputs(res, str(tmp_path / "c"), bench.DUMP_LIMIT)


def test_record_cache_is_keyed_on_the_generating_sources(tmp_path, monkeypatch):
    """A cached block is read only by the version of the scenario generator, record layout and planners that
    wrote it: changing one of them changes the cache directory."""
    import shutil
    sys.path.insert(0, ROOT)
    import bench
    for d in ("p-dmpc_b200", "include", "oracle"):
        shutil.copytree(os.path.join(ROOT, d), tmp_path / d, ignore=shutil.ignore_patterns("*.so", "__pycache__"))
    shutil.copy(os.path.join(ROOT, "bench.py"), tmp_path / "bench.py")
    monkeypatch.setattr(bench, "ROOT", str(tmp_path))
    v0 = bench.records_version()
    assert v0 == os.path.basename(bench.RECORD_CACHE)
    for f in ("p-dmpc_b200/scenario.py", "p-dmpc_b200/records.py", "p-dmpc_b200/csrc/pdmpc_tiles.cuh", "oracle/pdmpc_oracle.c"):
        with open(tmp_path / f, "a") as fh:
            fh.write("\n")
        v1 = bench.records_version()
        assert v1 != v0, f
        v0 = v1
