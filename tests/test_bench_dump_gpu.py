"""bench.py --dump-outputs: the dumped result of the last timed step equals the oracle's reduce_by_key of the
same seeded input, row for row, so two builds can be compared through their dumps."""
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest

from oracle import oracle as O

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _from_halves(a):
    return (a[:, 0].astype(np.uint64) << np.uint64(32)) | a[:, 1].astype(np.uint64)


def test_dump_outputs_match_oracle():
    n, D, M, R = 2_000_000, 50_000, 8, 8
    with tempfile.TemporaryDirectory() as d:
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--rows", str(n),
                              "--distinct", str(D), "--no-e2e", "--no-cpu", "--dump-outputs", d],
                             capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-4000:]
        got = {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d)}
    assert sorted(got) == ["keys", "partition_rows", "sums"]
    assert all(a.dtype == np.float64 for a in got.values())
    keys, sums = _from_halves(got["keys"]), _from_halves(got["sums"])
    k, v = O.gen_uniform(0, n, D, 1, 2)
    want = O.shuffle("sum", k, v, M, R)
    assert got["partition_rows"].tolist() == [len(p["keys"]) for p in want]
    o = np.concatenate([p["keys"][np.argsort(p["keys"], kind="stable")] for p in want])
    c = np.concatenate([p["combined"][np.argsort(p["keys"], kind="stable")] for p in want])
    assert np.array_equal(keys, o) and np.array_equal(sums, c)
