"""bench.py contract on the CPU: the reference arm (--impl reference) prints ONE JSON line with the agreed keys, and the
product arm refuses to run without a CUDA device (no CPU fallback)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "descriptor_pairs_per_sec" and d["unit"] == "pairs/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["value"] > 0 and d["ms_per_step"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert set(d["config"]) == {"workload", "F", "k", "ratio", "pairs_per_step"} and d["config"]["workload"].startswith("C2")
    assert "sample" in d["cpu_baseline"] and d["cpu_baseline"]["cores"] == os.cpu_count()
    assert d["reference_exhaustive_blas"]["value"] > 0
    if "reference_default_engine" in d:   # needs the OpenCV python module
        assert 0.0 < d["reference_default_engine"]["recall_at_k_vs_exact"] <= 1.0


def test_reference_arm_uses_all_cores_under_torchrun_env():
    """torch.distributed.run exports OMP_NUM_THREADS=1; the reference arm must still use every host core, and at
    N > 1 it times the config the GPU arm runs there (C3)."""
    env = dict(os.environ, RANK="0", WORLD_SIZE="2", LOCAL_RANK="0", OMP_NUM_THREADS="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                        "--warmup", "1"], capture_output=True, text=True, timeout=900, cwd=ROOT, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][0])
    assert d["cpu_baseline"]["cores"] == os.cpu_count() and d["config"]["workload"].startswith("C3") and d["scaling"] == "strong"


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                       capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_steps_must_be_positive():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True,
                       timeout=120, cwd=ROOT)
    assert r.returncode == 2 and "--steps must be at least 1" in r.stderr


def test_pairwise_shares_merge_into_one_csr():
    """--dump-outputs on several ranks: the block-cyclic shares of the pair list (as multigpu.exchange_pairwise_lists
    returns them) merge into the CSR one rank computes."""
    import numpy as np

    import bench

    n, world = 6, 4
    rng = np.random.default_rng(1)
    counts = np.zeros(n * n, np.int64)
    pairs = [i + j * n for j in range(n) for i in range(j)]          # column-major pair list
    counts[pairs] = rng.integers(0, 4, len(pairs))
    pp = np.concatenate([[0], np.cumsum(counts)])
    rows = rng.integers(1, 1000, (pp[-1], 2)).astype(np.uint32)
    met = rng.random(pp[-1])
    share_counts = np.zeros((world, n * n), np.int64)
    for o, c in enumerate(pairs):
        share_counts[o % world, c] = counts[c]
    m_max = int(share_counts.sum(1).max())
    rows_all, met_all = np.zeros((world, m_max, 2), np.uint32), np.zeros((world, m_max))
    for r in range(world):
        mine = np.concatenate([np.arange(pp[c], pp[c + 1]) for c in range(n * n) if share_counts[r, c]] or [[]]).astype(int)
        rows_all[r, :len(mine)], met_all[r, :len(mine)] = rows[mine], met[mine]
    got_pp, got_rows, got_met = bench.pairwise_csr_of_shares(share_counts, rows_all, met_all)
    assert np.array_equal(got_pp, pp) and np.array_equal(got_rows, rows) and np.array_equal(got_met, met)


def test_product_arm_needs_a_gpu():
    import torch

    if torch.cuda.is_available():
        import pytest

        pytest.skip("GPU present")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1"], capture_output=True, text=True,
                       timeout=300, cwd=ROOT)
    assert r.returncode != 0 and "no CUDA device" in (r.stderr + r.stdout)
