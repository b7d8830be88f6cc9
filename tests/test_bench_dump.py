"""bench.py --dump-outputs: the decision records of the last timed step, one .npy per field, exact in float32 / float64."""
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_round_trips_every_field_exactly(tmp_path):
    import bench
    from cordum_b200 import wire

    rng = np.random.default_rng(5)
    rec = np.zeros(1000, dtype=wire.DECISION_DTYPE)
    for f in ("decision", "sched_decision", "flags", "route_status", "reason_code"):
        rec[f] = rng.integers(0, 256, len(rec))
    rec["rule_idx"] = rng.integers(-1, 4096, len(rec))
    rec["worker_slot"] = rng.integers(-1, 65536, len(rec))
    rec["rule_idx"][:2] = (np.iinfo(np.int32).min, np.iinfo(np.int32).max)   # float32 would round these
    rec["worker_slot"][:2] = (np.iinfo(np.int32).max, np.iinfo(np.int32).min)
    bench.dump_outputs(str(tmp_path), rec, 0, 1)
    assert sorted(os.listdir(tmp_path)) == sorted(f + ".npy" for f in bench.DECISION_FIELDS)
    for f in bench.DECISION_FIELDS:
        a = np.load(tmp_path / (f + ".npy"))
        assert a.dtype in (np.float32, np.float64) and a.shape == rec.shape
        assert np.array_equal(a.astype(np.int64), rec[f].astype(np.int64)), f
    # 1M jobs (config 3, the benchmark's workload) stay under 64 MB in all
    per_job = sum(np.load(tmp_path / (f + ".npy")).itemsize for f in bench.DECISION_FIELDS)
    assert per_job * 1_000_000 <= 64 << 20

    bench.dump_outputs(str(tmp_path / "sharded"), rec, 1, 2)
    assert sorted(os.listdir(tmp_path / "sharded")) == sorted(f + ".rank1.npy" for f in bench.DECISION_FIELDS)


def test_bench_rejects_zero_steps_and_dumping_the_reference_leg(tmp_path):
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path)]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True, timeout=120)
        assert r.returncode == 2 and "error" in r.stderr, (extra, r.stderr)
