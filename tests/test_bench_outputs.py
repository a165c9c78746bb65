"""bench.py --dump-outputs: the headline run writes the result of its last timed MSM, and that result is the oracle's
(sum k_i s_i)*G for the benchmark's seeded inputs, so two builds can be compared output for output."""
import json
import os
import random
import subprocess
import sys

import numpy as np
import pytest

from oracle import noble_ref as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_rejected_outside_the_headline_run(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert out.returncode == 2 and "--dump-outputs" in out.stderr
    assert os.listdir(tmp_path) == []


@pytest.mark.gpu
def test_dump_outputs_match_oracle(tmp_path):
    logn, steps = 12, 3
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--logn", str(logn), "--steps", str(steps), "--warmup", "1",
                          "--no-cpu-baseline", "--no-fixed-base", "--no-pipelined", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads(out.stdout.strip().splitlines()[-1])
    assert d["steps"] == steps and d["e2e"]["steps"] == steps and d["config"]["terms"] == 1 << logn
    assert sorted(os.listdir(tmp_path)) == ["msm_affine_xy_limbs.npy", "msm_is_infinity.npy"]
    xy = np.load(tmp_path / "msm_affine_xy_limbs.npy")
    inf = np.load(tmp_path / "msm_is_infinity.npy")
    assert xy.dtype == np.float64 and xy.shape == (2, 12) and inf.dtype == np.float64 and inf.shape == (1,)
    x, y = (sum(int(v) << (32 * i) for i, v in enumerate(row)) for row in xy)
    # bench.make_terms on rank 0: points k_i*G and scalars s_i drawn from random.Random(1000)
    P = R.CURVES["bls12_381_G1"]
    order = P.Fn.ORDER
    rnd = random.Random(1000)
    ks = [rnd.randrange(1, order) for _ in range(1 << logn)]
    sc = [rnd.randrange(order) for _ in range(1 << logn)]
    exp = P.BASE.multiplyUnsafe(sum(k * s for k, s in zip(ks, sc)) % order).toAffine()
    assert (x, y, int(inf[0])) == (exp["x"], exp["y"], 0)
