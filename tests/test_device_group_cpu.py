"""Device groups (single-process multi-GPU matching) without a GPU: aps_group_create fails loudly (no CPU fallback), the
host mirror rejects input.apsGPUs together with shard= and malformed device lists, and the batched MEX gateway checks
its trailing `gpus` argument before any device is touched (under the mex shim)."""
import ctypes
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _no_gpu_with_library(aps):
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present: covered by tests/test_gpu_device_group.py")
    if not os.path.exists(aps.library_path()):
        pytest.skip("libapsmatch.so not built")


def test_group_create_without_gpu_is_nogpu(aps):
    _no_gpu_with_library(aps)
    L = aps._lib.lib()
    devs = (ctypes.c_int * 2)(0, 1)
    h = ctypes.c_void_p()
    assert L.aps_group_create(devs, 2, ctypes.byref(h)) == 6          # APS_ERR_NOGPU
    assert L.aps_error_id().decode() == "apsmatch:nogpu"
    assert not h.value
    with pytest.raises(aps.ApsError) as e:
        aps.DeviceGroup([0, 1])
    assert e.value.code == 6 and e.value.identifier == "apsmatch:nogpu"


def test_group_create_rejects_malformed_lists_before_looking_for_a_device(aps):
    if not os.path.exists(aps.library_path()):
        pytest.skip("libapsmatch.so not built")
    L = aps._lib.lib()
    h = ctypes.c_void_p()
    assert L.aps_group_create(None, 0, ctypes.byref(h)) == 1           # APS_ERR_ARGS
    assert L.aps_group_create((ctypes.c_int * 2)(1, 1), 2, ctypes.byref(h)) == 1
    assert L.aps_group_create((ctypes.c_int * 2)(0, -1), 2, ctypes.byref(h)) == 1
    assert L.aps_group_size(None) == 0 and not L.aps_group_ctx(None, 0)


def test_host_rejects_apsGPUs_with_shard(aps):
    import numpy as np

    desc = [np.zeros((4, 8), np.float32)] * 2
    inp = {"Matchingthreshold": 1.5, "Ratiothreshold": 0.6, "apsGPUs": [1, 2]}
    with pytest.raises(ValueError, match="shard"):
        aps.featureMatchingPairwise(inp, desc, 2, shard=(0, 2))
    with pytest.raises(ValueError, match="shard"):
        aps.featureMatchingPairwise(dict(inp, apsGPUs=[1]), desc, 2, shard=(1, 2))


@pytest.mark.parametrize("gpus", [[0, 1], [1, 1.5], [2, 2], [1, float("nan")], [-1]])
def test_host_rejects_malformed_apsGPUs(aps, gpus):
    import numpy as np

    desc = [np.zeros((4, 8), np.float32)] * 2
    with pytest.raises(ValueError, match="apsGPUs"):
        aps.featureMatchingGlobal({"k": 4, "Ratiothreshold": 0.6, "apsGPUs": gpus}, desc, 2)
    with pytest.raises(ValueError, match="apsGPUs"):
        aps.featureMatchingPairwise({"Matchingthreshold": 1.5, "Ratiothreshold": 0.6, "apsGPUs": gpus}, desc, 2)


def test_gateway_gpus_argument_checks(aps):
    _no_gpu_with_library(aps)
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "mex"), "shimcheck"], check=True, capture_output=True)
    r = subprocess.run([os.path.join(ROOT, "mex", "_build", "gate_batched"), "gpus"], capture_output=True, text=True)
    assert r.returncode == 0 and "OK" in r.stdout, r.stdout + r.stderr
