"""Build guard for the per-tile cycle accounting of k_knn_tc (-DAPS_TC_TILE_CLOCKS, profiles/tile_clocks.py): the
measurement variant still compiles for sm_100a and exports its read-back entry, and the default build is the kernel
without any of it -- the same SASS, instruction for instruction, as the source with the instrumentation cut out."""
import os
import re
import shutil
import subprocess

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "..", "automaticpanoramicimagestitching-autopanostitch-matlab_b200", "csrc")
SRC = os.path.join(CSRC, "aps_knn_tc.cu")


def _compile(tmp_path, src, name, *defines):
    nvcc = shutil.which("nvcc")
    if nvcc is None or shutil.which("cuobjdump") is None or shutil.which("nm") is None:
        pytest.skip("nvcc / cuobjdump / nm not available")
    obj = tmp_path / name
    r = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-I", CSRC, *defines,
                        "-c", "-o", str(obj), str(src)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-4000:]
    return obj


def _kernel_sass(obj):
    """SASS of every k_knn_tc instantiation, keyed by its template arguments (the anonymous-namespace hash in the
    mangled name depends on the file's path, so it is not part of the key)."""
    out = subprocess.run(["cuobjdump", "-sass", str(obj)], capture_output=True, text=True, check=True).stdout
    funcs, cur = {}, None
    for line in out.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            k = re.search(r"k_knn_tcI(\S*?)EEEv", m.group(1))
            cur = k.group(1) if k else None
            if cur:
                funcs[cur] = []
            continue
        if cur and re.search(r"/\*[0-9a-f]{4,}\*/", line):
            funcs[cur].append(re.sub(r"\s+", " ", line.split(";")[0]).strip())
    return funcs


def _strip_instrumentation(text):
    """Drops the `#ifdef APS_TC_TILE_CLOCKS` blocks (keeping their `#else` side) and every APS_CLK(...) statement."""
    out, depth, mode = [], 0, None  # mode: None outside, "drop" / "keep" inside a clocks block
    for line in text.splitlines(keepends=True):
        s = line.strip()
        if mode is None and s == "#ifdef APS_TC_TILE_CLOCKS":
            mode, depth = "drop", 0
            continue
        if mode is not None:
            if s.startswith("#if"):
                depth += 1
            elif s.startswith("#endif"):
                if depth == 0:
                    mode = None
                    continue
                depth -= 1
            elif s.startswith("#else") and depth == 0:
                mode = "keep"
                continue
            if mode == "drop" or s.startswith("#define APS_CLK"):  # nothing uses the macro once its uses are cut
                continue
        out.append(line)
    text = "".join(out)
    res, i = [], 0
    while True:
        j = text.find("APS_CLK(", i)
        if j < 0:
            res.append(text[i:])
            break
        res.append(text[i:j])
        k, depth = j + len("APS_CLK("), 1
        while depth:
            depth += {"(": 1, ")": -1}.get(text[k], 0)
            k += 1
        i = k
    return "".join(res)


def test_tile_clock_variant_compiles_and_exports_its_reader(tmp_path):
    obj = _compile(tmp_path, SRC, "clk.o", "-DAPS_TC_TILE_CLOCKS")
    assert " T aps_debug_tile_clocks" in subprocess.run(["nm", str(obj)], capture_output=True, text=True).stdout


def test_default_build_is_the_kernel_without_instrumentation(tmp_path):
    with open(SRC) as f:
        text = f.read()
    stripped = _strip_instrumentation(text)
    assert "#ifdef APS_TC_TILE_CLOCKS" not in stripped and "clock()" not in stripped
    bare = tmp_path / "aps_knn_tc.cu"
    bare.write_text(stripped)
    default = _kernel_sass(_compile(tmp_path, SRC, "default.o"))
    reference = _kernel_sass(_compile(tmp_path, bare, "bare.o"))
    assert len(default) >= 14 and sorted(default) == sorted(reference)
    for k in default:
        assert default[k] == reference[k], f"k_knn_tc<{k}> differs from the kernel without the tile clocks"
