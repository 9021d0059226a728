"""bench.py: the reference arm prints one JSON line with the keys every bench line carries (CPU);
--dump-outputs writes the solutions of the last timed step, within its size budget and identical
from run to run (GPU)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bench_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference",
                          "--workload", "C1", "--steps", "2", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = [l for l in out.stdout.splitlines() if l.startswith("{")][-1]
    d = json.loads(line)
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
              "scaling", "vs_baseline", "dtype", "data", "config", "impl", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["dtype"] == "f64" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["unit"] == "it/s"
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] == 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["config"]["workload"].startswith("C1")


def test_bench_reference_arm_nonzero_rank_exits_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference",
                          "--workload", "C1", "--steps", "1", "--warmup", "0", "--gpus", "2"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and "{" not in out.stdout


def test_dump_budget_samples_large_outputs_deterministically():
    import bench
    # C5: three solves, x of length n = 1e6 and z of length m = 2.002e6 each
    outs = {f"solve{k}_{v}": np.zeros(1_000_000 if v == "x" else 2_002_000) for k in (1, 2, 3) for v in "xz"}
    fitted = bench.fit_dump_budget(outs)
    assert sum(a.nbytes + 4096 for a in fitted.values()) <= bench.DUMP_BUDGET_BYTES
    assert fitted["solve1_x"].size == 1_000_000 and 0 < fitted["solve1_z"].size < 2_002_000
    small = {"a": np.arange(10.0), "b": np.arange(1000, dtype=np.float32)}
    f1 = bench.fit_dump_budget(small, budget=2 * 4096 + 2 * 8 * 100)
    f2 = bench.fit_dump_budget(small, budget=2 * 4096 + 2 * 8 * 100)
    assert all(a.dtype == np.float64 for a in f1.values())
    assert np.array_equal(f1["a"], small["a"])
    b = f1["b"]
    assert b.size == 100 and np.all(np.diff(b) > 0) and np.all(np.isin(b, small["b"]))
    assert np.array_equal(b, f2["b"])


def test_replay_inputs_round_trip(tmp_path):
    import bench
    rng = np.random.default_rng(0)
    keys = ("w", "soc_eta", "soc_d", "soc_u", "soc_v", "psd_R")
    replay = [dict(state={k: rng.standard_normal(3 if k == "w" else 0) for k in keys},
                   rhs=[(rng.standard_normal(2), rng.standard_normal(3)) for _ in range(3)]) for _ in range(4)]
    path = str(tmp_path / "inputs")
    bench.save_replay(path, "C1", 2, 3, [1, 5, 8, 9], replay)
    ids, back = bench.load_replay(path, "C1", 2, 3)
    assert ids == [1, 5, 8, 9] and len(back) == 4
    for a, b in zip(replay, back):
        assert a["state"].keys() == b["state"].keys()
        assert all(np.array_equal(a["state"][k], b["state"][k]) for k in keys)
        assert len(b["rhs"]) == 3
        assert all(np.array_equal(x, y) for ra, rb in zip(a["rhs"], b["rhs"]) for x, y in zip(ra, rb))
    with pytest.raises(SystemExit, match="not of C2"):
        bench.load_replay(path, "C2", 2, 3)


@pytest.mark.gpu
def test_bench_dump_outputs_are_reproducible(tmp_path):
    """Two runs share --replay-inputs: the first stores its replayed systems, the second replays the
    stored ones.  The dumps must be identical, and each dumped solution must be the CPU oracle's
    solution of the last timed step's system (step warmup + steps - 1, modulo the replayed systems)."""
    import bench
    steps, warmup = 2, 3
    inputs = tmp_path / "inputs.npz"
    lines, dumps = [], []
    for run in ("a", "b"):
        d = tmp_path / run
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "C1", "--steps", str(steps),
                              "--warmup", str(warmup), "--no-cpu-baseline", "--dump-outputs", str(d),
                              "--replay-inputs", str(inputs)],
                             capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        lines.append(json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1]))
        dumps.append({f: np.load(d / f) for f in sorted(os.listdir(d))})
    line = lines[0]
    assert line["steps"] == steps and line["parity"]["ok"]
    n, m = line["config"]["n"], line["config"]["m"]
    assert sorted(dumps[0]) == sorted(f"solve{k}_{v}.npy" for k in (1, 2, 3) for v in "xz")
    for name, a in dumps[0].items():
        assert a.dtype == np.float64 and a.shape == ((n,) if name.endswith("_x.npy") else (m,))
        assert np.all(np.isfinite(a)) and np.array_equal(a, dumps[1][name]), name
    _, replay = bench.load_replay(str(inputs), "C1", n, m)
    cpu = {}
    bench.cpu_full_step(bench.make_problem("C1"), replay[(warmup + steps - 1) % len(replay)], cpu)
    assert "error" not in cpu and cpu["ok"]
    for k, c in enumerate(cpu["sols"], 1):
        g = np.concatenate([dumps[0][f"solve{k}_x.npy"], dumps[0][f"solve{k}_z.npy"]])
        assert np.abs(g - c).max() <= 1e-6 * np.abs(c).max(), k
