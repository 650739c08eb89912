"""bench.py's --steps and --dump-outputs: the number of timed steps is the one asked for, and the dumped Gt values of the
last timed step equal the C oracle's pairings of the same seeded inputs (the point generator's SplitMix64 scalars)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import util

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SEED = 0x5EED5EED          # bench.py's synthetic-input seed


def _bench(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=900, cwd=ROOT)


def test_bench_rejects_bad_arguments(tmp_path):
    for args in (["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", str(tmp_path / "d")]):
        r = _bench(*args)
        assert r.returncode == 2 and "error:" in r.stderr, (args, r.stderr[-500:])
    assert not any(tmp_path.iterdir())


@pytest.mark.gpu
def test_bench_steps_and_dumped_outputs(coracle, tmp_path):
    import bench
    log2 = 16
    common = ["--gpus", "1", "--warmup", "1", "--log2-batch", str(log2), "--no-configs", "--no-cpu-baseline"]
    runs = {}
    for steps in (1, 3):
        r = _bench(*common, "--steps", str(steps), "--dump-outputs", str(tmp_path / str(steps)))
        assert r.returncode == 0, r.stderr[-2000:]
        runs[steps] = json.loads(r.stdout)
        assert runs[steps]["steps"] == steps and runs[steps]["e2e"]["steps"] == steps
    assert runs[1]["gpu_launches"] > 0 and runs[3]["gpu_launches"] == 3 * runs[1]["gpu_launches"]

    gt = np.load(tmp_path / "3" / "gt.npy")
    assert np.array_equal(gt, np.load(tmp_path / "1" / "gt.npy"))           # same inputs, same outputs
    rows = bench.dump_rows(1 << log2)
    assert len(rows) == bench.DUMP_ROWS < 1 << log2 and np.array_equal(rows, np.unique(rows))
    assert gt.dtype == np.float64 and gt.shape == (len(rows), 144) and gt.nbytes <= 64 << 20
    limbs = gt.astype(np.uint64)
    assert np.array_equal(limbs.astype(np.float64), gt) and int(limbs.max()) < 1 << 32
    got = limbs[:, 0::2] | (limbs[:, 1::2] << np.uint64(32))
    pick = np.arange(0, len(rows), len(rows) // 256)
    ab = [util.scalars_for(SEED, int(i), 1) for i in rows[pick]]
    g1, i1 = coracle.g1_mul_batch(util.scalar_matrix([a[0] for a, _ in ab]))
    g2, i2 = coracle.g2_mul_batch(util.scalar_matrix([b[0] for _, b in ab]))
    assert np.array_equal(got[pick], coracle.pairing_batch(g1, i1, g2, i2))
