"""bench.py --dump-outputs on the GPU: the match lists dumped from the last timed step equal what the public calls return
for the same synthetic inputs, in float64 and within bench.DUMP_LIMIT."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
@pytest.mark.parametrize("config", ["c2", "c5"])
def test_dump_outputs_equal_the_public_call(aps, config, tmp_path):
    import bench

    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", config, "--steps", "2",
                        "--no-cpu-baseline", "--no-extra", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    got = {f: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    assert all(a.dtype == np.float64 for a in got.values())
    assert sum(os.path.getsize(tmp_path / f) for f in got) <= bench.DUMP_LIMIT
    cid, kind, _ = bench.CONFIGS[config]
    desc, c = aps.synth.make_config(cid)
    n = len(desc)
    if kind == "pairwise":
        pp, rows, met = aps.featureMatchingPairwise(bench.C5_INPUT, desc, n, csr=True)
        assert sorted(got) == ["matches.npy", "metric.npy", "pair_ptr.npy"]
        assert np.array_equal(got["metric.npy"], met)
    else:
        cells = aps.featureMatchingGlobal({"k": bench.KNN, "Ratiothreshold": c["ratio"], "BFMatch": 1}, desc, n)
        cells = [cells[cc % n][cc // n] for cc in range(n * n)]      # column-major cell order of pair_ptr
        pp = np.concatenate([[0], np.cumsum([m.shape[0] for m in cells])])
        rows = np.concatenate([m for m in cells if m.shape[0]])
        assert sorted(got) == ["matches.npy", "pair_ptr.npy"]
    assert pp[-1] > 0
    assert np.array_equal(got["pair_ptr.npy"], pp) and np.array_equal(got["matches.npy"], rows)
