"""bench.py --dump-outputs: what the timed path returned in its last step, written as .npy files of bounded size so that two builds
run with the same arguments can be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_is_bounded_and_samples_problems_with_a_fixed_seed(tmp_path):
    import bench
    B = 4096
    rng = np.random.default_rng(3)
    arrays = dict(xp=rng.standard_normal((B, 81, 4)), np=rng.standard_normal((B, 81, 12)), lp=rng.standard_normal((B, 81, 5)),
                  sl=rng.standard_normal((B, 81, 3)), exitflag=np.ones(B, np.int32), iters=np.arange(B, dtype=np.int32))
    arrays["xp"] = np.concatenate([arrays["xp"]] * 3, axis=2)        # 8.7 KB more per problem: over 64 MB at this batch
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == sorted([k + ".npy" for k in arrays] + ["problem.npy"])
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64 * 10**6
    idx = np.load(tmp_path / "a" / "problem.npy")
    assert 0 < len(idx) < B and np.all(np.diff(idx) > 0)
    for f in files:
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype == np.float64 and np.array_equal(a, b)
    assert np.array_equal(np.load(tmp_path / "a" / "iters.npy"), idx)
    assert np.array_equal(np.load(tmp_path / "a" / "xp.npy"), arrays["xp"][idx.astype(int)])
    small = {k: v[:10] for k, v in arrays.items()}
    bench.dump_outputs(str(tmp_path / "c"), small)
    assert np.array_equal(np.load(tmp_path / "c" / "problem.npy"), np.arange(10))


@pytest.mark.gpu
def test_bench_dumps_the_outputs_of_its_last_step(tmp_path):
    """The headline arm at a small batch: the dumped outputs (C-ABI layout, problem-major) are the solutions the library returns
    for the same seeded batch through the host-pointer call."""
    from obca_b200 import parking, scenarios
    B, out = 64, tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--batch", str(B), "--steps", "2", "--warmup", "1", "--no-cpu",
                        "--dump-outputs", str(out)], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout)
    assert line["steps"] == 2 and line["config"]["batch_per_gpu"] == B
    d = {f[:-4]: np.load(out / f) for f in os.listdir(out)}
    assert sorted(d) == sorted(["problem", "xp", "up", "ts", "lp", "np", "sl", "exitflag", "iters", "kkt_err"])
    assert all(a.dtype == np.float64 and a.shape[0] == B for a in d.values())
    assert np.array_equal(d["problem"], np.arange(B)) and d["exitflag"].sum() == round(line["config"]["converged_frac"] * B)
    sc = scenarios.reverse_parking_batch(B, 80, seed=0)
    ref = parking.parking_solve_batch(sc["x0"], sc["xF"], 80, sc["Ts"], sc["L"], sc["ego"], sc["XYbounds"], sc["nOb"], sc["vOb"],
                                      sc["A"], sc["b"], sc["rx"], sc["ry"], sc["ryaw"], 0, sc["xWS"], sc["uWS"])
    assert np.array_equal(d["exitflag"], ref["exitflag"]) and np.array_equal(d["iters"], ref["iters"])
    T = lambda a: np.transpose(a, (0, 2, 1))
    for k in ("xp", "up", "lp", "np", "sl"):
        assert np.abs(d[k] - T(ref[k])).max() < 1e-8, k
    assert np.abs(d["ts"] - ref["ts"]).max() < 1e-8
