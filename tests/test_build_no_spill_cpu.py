"""Build guard for the tensor-core kNN kernel: every k_knn_tc instantiation compiles for sm_100a without local-memory
spills and with the register allocation its setmaxnreg split was computed for (168 per thread for 384 threads, 96 for
the 640-thread short-sweep variant; a smaller allocation would leave setmaxnreg.inc waiting for registers)."""
import os
import re
import shutil
import subprocess

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "..", "automaticpanoramicimagestitching-autopanostitch-matlab_b200", "csrc")


@pytest.fixture(scope="module")
def ptxas_report(tmp_path_factory):
    nvcc = shutil.which("nvcc")
    if nvcc is None:
        pytest.skip("nvcc is not available")
    obj = tmp_path_factory.mktemp("knn_tc") / "aps_knn_tc.o"
    r = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v",
                        "-c", "-o", str(obj), os.path.join(CSRC, "aps_knn_tc.cu")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-4000:]
    entries = {}
    name = None
    for line in r.stderr.splitlines():
        m = re.search(r"Compiling entry function '(\S*k_knn_tc\S*)'", line)
        if m:
            name, entries[m.group(1)] = m.group(1), {}
            continue
        if name is None:
            continue
        m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m:
            entries[name].update(stack=int(m.group(1)), spill_st=int(m.group(2)), spill_ld=int(m.group(3)))
        m = re.search(r"Used (\d+) registers", line)
        if m:
            entries[name]["regs"] = int(m.group(1))
            name = None
    return entries


def test_every_instantiation_is_reported(ptxas_report):
    assert len(ptxas_report) >= 14, sorted(ptxas_report)
    assert all({"stack", "spill_st", "spill_ld", "regs"} <= set(v) for v in ptxas_report.values()), ptxas_report


def test_no_spills_and_no_stack(ptxas_report):
    bad = {k: v for k, v in ptxas_report.items() if v["stack"] or v["spill_st"] or v["spill_ld"]}
    assert not bad, bad


def test_launch_allocation_matches_the_register_split(ptxas_report):
    for name, v in ptxas_report.items():
        short_sweep = "ELi3ELi2E" in name  # KCT == 3, CS == 2: 20 warps
        assert v["regs"] == (96 if short_sweep else 168), (name, v)
