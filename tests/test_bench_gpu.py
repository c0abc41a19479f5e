"""bench.py on the device at a small size: the outputs it dumps are those of the timed search, equal to the CPU
oracle's plans of the same records."""
import dataclasses
import json
import os
import subprocess
import sys
import types

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_dump_outputs_equal_the_oracle_on_the_same_records(built, tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--scenarios", "8", "--sim-steps", "6",
                          "--steps", "2", "--warmup", "1", "--no-cache", "--gen-workers", "1",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    n = line["config"]["searches_per_step_per_gpu"]
    assert n == 8 * 6 * 20
    assert line["steps"] == 2                                         # the number of CUDA-event-timed steps
    assert abs(line["value"] - n * 2 / (line["ms_per_step"] * 2e-3)) < 1e-6 * line["value"]

    sys.path.insert(0, ROOT)
    import bench
    from oracle import oracle_py, parity
    from pdmpc_b200.mpa import get_mpa
    from pdmpc_b200.records import BatchResult
    args = types.SimpleNamespace(no_cache=True, mpa="triple_speed", vehicles=20, sim_steps=6)
    batch, _levels, _ts = bench.get_records(args, [0], "oracle", 0, 1)
    mpa = get_mpa("triple_speed", non_convex=True)
    ref = oracle_py.plan_batch(mpa, batch, 4)
    ref_valid = oracle_py.plan_batch(mpa, batch, 4, hash_valid_pops_only=True)

    d = {f[:-4]: np.load(os.path.join(tmp_path, f)) for f in os.listdir(tmp_path)}
    assert all(a.dtype == np.float64 and np.isfinite(a).all() for a in d.values())
    assert np.array_equal(d.pop("rows"), np.arange(n))
    hi, lo = d.pop("pop_hash_hi").astype(np.uint64), d.pop("pop_hash_lo").astype(np.uint64)
    got = BatchResult.empty(n, mpa.Hp)
    got.pop_hash[:] = (hi << np.uint64(32)) | lo
    for f in dataclasses.fields(got):
        if f.name in d:
            getattr(got, f.name)[...] = d.pop(f.name)
    assert not d
    ex = got.is_exhausted.astype(bool)
    # the dump writes the NaN plans of exhausted searches as 0
    assert (got.y_predicted[ex] == 0).all() and (got.g_path[ex] == 0).all() and (got.h_path[ex] == 0).all()
    got.y_predicted[ex] = got.g_path[ex] = got.h_path[ex] = np.nan
    parity.compare(got, ref, skip=("pop_hash",))
    # the pops the hash covers depend on the launch shape the library picks (pdmpc_set_variant, include/pdmpc_b200.h)
    assert ((got.pop_hash == ref.pop_hash) | (got.pop_hash == ref_valid.pop_hash)).all()
