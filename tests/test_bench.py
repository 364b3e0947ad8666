"""bench.py's host-side pieces (no GPU): argument checks and --dump-outputs' writer."""
import os
import subprocess
import sys

import numpy as np

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _outputs(n):
    rng = np.random.default_rng(1)
    return {"cfg4": {"z": rng.normal(size=n), "idx": rng.integers(0, 801, size=(n, 3)).astype(np.int32), "cz": rng.random(n)},
            "cfg5": {"z": rng.normal(size=2 * n), "adjusted_z": rng.normal(size=2 * n)}}


def _read(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_dump_outputs_writes_every_array_in_float64(tmp_path):
    out = _outputs(50)
    bench.dump_outputs(out, str(tmp_path))
    got = _read(str(tmp_path))
    assert sorted(got) == ["cfg4_cz", "cfg4_idx", "cfg4_z", "cfg5_adjusted_z", "cfg5_z"]
    for cfg, res in out.items():
        for name, v in res.items():
            a = got[f"{cfg}_{name}"]
            assert a.dtype == np.float64 and np.array_equal(a, v)


def test_dump_outputs_samples_the_same_rows_under_a_byte_budget(tmp_path):
    out = _outputs(1000)
    budget = 20_000  # the arrays take 72 000 bytes in float64, 96 000 with the sampled rows (8 bytes a row)
    a, b = str(tmp_path / "a"), str(tmp_path / "b")
    bench.dump_outputs(out, a, max_bytes=budget)
    bench.dump_outputs(out, b, max_bytes=budget)
    got, again = _read(a), _read(b)
    assert sorted(got) == sorted(again) and all(np.array_equal(got[k], again[k]) for k in got)  # fixed, seeded sample
    payload = sum(v.nbytes for v in got.values())
    assert 0.9 * budget < payload <= budget
    for cfg, res in out.items():
        rows = got[f"{cfg}_genes"].astype(np.int64)
        assert np.all(np.diff(rows) > 0) and rows[0] >= 0 and rows[-1] < len(res["z"])
        for name, v in res.items():
            assert np.array_equal(got[f"{cfg}_{name}"], v[rows])


def test_step_count_and_reference_dump_are_checked():
    for argv in (["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "x"]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + argv, capture_output=True, text=True)
        assert r.returncode == 2 and "error:" in r.stderr, argv
