"""ctypes binding of libapsmatch.so -- exactly the symbols include/apsmatch.h declares."""
from __future__ import annotations

import ctypes as C
import glob
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libapsmatch.so")

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared"]

APS_COL_MAJOR, APS_ROW_MAJOR = 0, 1
APS_F32, APS_U8 = 0, 1

ERR_NAMES = {1: "APS_ERR_ARGS", 2: "APS_ERR_TYPE", 3: "APS_ERR_K", 4: "APS_ERR_DIM", 5: "APS_ERR_BF",
             6: "APS_ERR_NOGPU", 7: "APS_ERR_CUDA", 8: "APS_ERR_ALLOC", 9: "APS_ERR_METHOD"}


class ApsError(RuntimeError):
    """Raised for a non-zero status; `.identifier` is the MATLAB error id the reference would use."""

    def __init__(self, code, identifier, message):
        super().__init__(f"[{ERR_NAMES.get(code, code)}] {identifier + ': ' if identifier else ''}{message}")
        self.code, self.identifier, self.message = code, identifier, message


def library_path() -> str:
    return _SO


def sources():
    return sorted(glob.glob(os.path.join(_HERE, "csrc", "*.cu")))


def build_library(force: bool = False, verbose: bool = False) -> str:
    """nvcc-compiles csrc/*.cu for sm_100a into libapsmatch.so next to this file (in-tree): one object per
    translation unit (compiled in parallel, rebuilt only when the source or a header changed), then one link."""
    from concurrent.futures import ThreadPoolExecutor

    srcs = sources()
    hdrs = glob.glob(os.path.join(_HERE, "csrc", "*.cuh")) + [os.path.join(_HERE, "..", "include", "apsmatch.h")]
    objdir = os.path.join(_HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    hdr_time = max(os.path.getmtime(h) for h in hdrs)
    jobs = []
    for src in srcs:
        obj = os.path.join(objdir, os.path.basename(src)[:-3] + ".o")
        if force or not os.path.exists(obj) or os.path.getmtime(obj) < max(os.path.getmtime(src), hdr_time):
            jobs.append((src, obj))
    flags = [f for f in NVCC_FLAGS if f != "-shared"]

    def compile_one(job):
        cmd = ["nvcc"] + flags + (["-Xptxas", "-v"] if verbose else []) + ["-c", "-o", job[1], job[0]]
        subprocess.run(cmd, check=True)

    if jobs:
        with ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 1)) as ex:
            list(ex.map(compile_one, jobs))
    objs = [os.path.join(objdir, os.path.basename(s)[:-3] + ".o") for s in srcs]
    if jobs or not os.path.exists(_SO) or any(os.path.getmtime(_SO) < os.path.getmtime(o) for o in objs):
        subprocess.run(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", _SO] + objs, check=True)
    return _SO


_lib = None


def lib():
    """Loads libapsmatch.so.  No fallback: a missing library is an error."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_SO):
        raise ApsError(6, "apsmatch:nolib", f"{_SO} is missing: run __graft_entry__.build() (nvcc, sm_100a); "
                                            "there is no CPU fallback")
    L = C.CDLL(_SO)
    vp, i64, i32, dbl, cp = C.c_void_p, C.c_int64, C.c_int, C.c_double, C.c_char_p
    pp = C.POINTER(vp)
    sig = {
        "aps_ctx_create": (i32, [i32, pp]),
        "aps_ctx_destroy": (None, [vp]),
        "aps_ctx_set_stream": (i32, [vp, vp]),
        "aps_ctx_synchronize": (i32, [vp]),
        "aps_last_error": (cp, []),
        "aps_error_id": (cp, []),
        "aps_abi_version": (i32, []),
        "aps_ctx_set_float_engine": (i32, [vp, i32]),
        "aps_ctx_set_pairwise_epilogue": (i32, [vp, i32]),
        "aps_ctx_last_stats": (i32, [vp, C.POINTER(i64)]),
        "aps_ctx_first_pass_unproven": (i64, [vp]),
        "aps_ctx_set_pairwise_screen": (i32, [vp, i32]),
        "aps_ctx_pairwise_stats": (i32, [vp, C.POINTER(i64)]),
        "aps_ctx_enable_timing": (i32, [vp, i32]),
        "aps_ctx_tc_time": (i32, [vp, C.POINTER(dbl), C.POINTER(i64)]),
        "aps_launch_count": (i64, []),
        "aps_host_alloc": (vp, [C.c_size_t]),
        "aps_host_free": (None, [vp]),
        "aps_flann_knn": (i32, [vp, vp, i64, vp, i64, i32, i32, i32, i32, cp, i32, i32, vp, vp]),
        "aps_nearest2_hamming": (i32, [vp, vp, i64, vp, i64, i32, i32, vp, vp, vp]),
        "aps_nearest2_ssd": (i32, [vp, vp, i64, vp, i64, i32, i32, vp, vp, vp]),
        "aps_match_features": (i32, [vp, vp, i64, vp, i64, i32, i32, i32, dbl, dbl, i32, vp, vp, C.POINTER(i64)]),
        "aps_match_features_bits": (i32, [vp, vp, i64, vp, i64, i32, i32, dbl, dbl, i32, vp, vp, C.POINTER(i64)]),
        "aps_feature_matching_global": (i32, [vp, pp, C.POINTER(i64), i32, i32, i32, i32, i32, dbl, i32, pp]),
        "aps_feature_matching_pairwise": (i32, [vp, pp, C.POINTER(i64), i32, i32, i32, i32, dbl, dbl, pp]),
        "aps_feature_matching_pairwise_shard": (i32, [vp, pp, C.POINTER(i64), i32, i32, i32, i32, dbl, dbl, i32, i32, pp]),
        "aps_feature_matching_pairwise_sets": (i32, [vp, i32, C.POINTER(i32), pp, C.POINTER(i64), i32, i32, i32, dbl, dbl,
                                                     i32, i64, C.c_uint64, pp]),
        "aps_matchlist_n": (i32, [vp]),
        "aps_matchlist_total": (i64, [vp]),
        "aps_matchlist_pair_ptr": (C.POINTER(i64), [vp]),
        "aps_matchlist_rows": (C.POINTER(C.c_uint32), [vp]),
        "aps_matchlist_metric": (C.POINTER(dbl), [vp]),
        "aps_matchlist_free": (None, [vp]),
        "aps_select_partners": (i32, [vp, vp, i32, i32, vp, vp, C.POINTER(i64)]),
        "aps_select_partners_sets": (i32, [vp, i32, vp, vp, i32, vp, vp, vp]),
        "aps_ransac_sample_table": (i32, [vp, vp, i64, i64, C.c_uint64, vp]),
        "aps_image_matching_batch": (i32, [vp, i64, vp, vp, vp, dbl, dbl, i32, vp, i64, C.c_uint64, vp, vp, vp, vp, vp, vp]),
        "aps_image_matching": (i32, [vp, i32, vp, vp, vp, vp, vp, i64, dbl, dbl, i32, vp, i64, C.c_uint64, vp, vp, vp, vp,
                                     vp, vp, vp]),
        "aps_image_matching_sets": (i32, [vp, i32, vp, vp, vp, vp, vp, vp, vp, dbl, dbl, i32, vp, i64, C.c_uint64, vp,
                                          vp, vp, vp, vp, vp, vp]),
        "aps_gplan_create": (i32, [vp, C.POINTER(i64), i32, i32, i32, i32, pp]),
        "aps_gplan_destroy": (None, [vp]),
        "aps_gplan_total": (i64, [vp]),
        "aps_gplan_desc_device": (vp, [vp]),
        "aps_gplan_upload": (i32, [vp, pp, i32]),
        "aps_gplan_prepare": (i32, [vp]),
        "aps_gplan_knn": (i32, [vp, i64, i64]),
        "aps_gplan_filter": (i32, [vp, i64, i64, dbl]),
        "aps_gplan_records_device": (vp, [vp]),
        "aps_gplan_knn_idx_device": (vp, [vp]),
        "aps_gplan_knn_dist_device": (vp, [vp]),
        "aps_gplan_compact": (i32, [vp]),
        "aps_gplan_filter_mutual": (i32, [vp]),
        "aps_feature_matching_global_dev": (i32, [vp, vp, C.POINTER(i64), i32, i32, i32, i32, dbl, i32, pp]),
        "aps_feature_matching_global_sets": (i32, [vp, i32, C.POINTER(i32), pp, C.POINTER(i64), i32, i32, i32, i32, dbl,
                                                   i32, i32, pp]),
        "aps_gplan_download_knn": (i32, [vp, i64, i64, vp, vp]),
        "aps_gplan_download": (i32, [vp, pp]),
        "aps_gplan_pair_counts_device": (i32, [vp, pp]),
        "aps_pplan_create": (i32, [vp, C.POINTER(i64), i32, i32, i32, pp]),
        "aps_pplan_destroy": (None, [vp]),
        "aps_pplan_total": (i64, [vp]),
        "aps_pplan_desc_device": (vp, [vp]),
        "aps_pplan_upload": (i32, [vp, pp, i32]),
        "aps_pplan_prepare": (i32, [vp]),
        "aps_pplan_match": (i32, [vp, dbl, dbl, i32, i32, pp]),
        "aps_pplan_set_method": (i32, [vp, i32, i64, C.c_uint64]),
        "aps_pplan_subset_table": (i32, [vp, i32, vp]),
        "aps_group_create": (i32, [C.POINTER(i32), i32, pp]),
        "aps_group_destroy": (None, [vp]),
        "aps_group_size": (i32, [vp]),
        "aps_group_ctx": (vp, [vp, i32]),
        "aps_group_stage_times": (i32, [vp, i32, C.POINTER(dbl)]),
        "aps_debug_group_create_shared": (i32, [i32, i32, pp]),
        "aps_group_feature_matching_global": (i32, [vp, pp, C.POINTER(i64), i32, i32, i32, i32, i32, dbl, i32, pp]),
        "aps_group_feature_matching_pairwise": (i32, [vp, pp, C.POINTER(i64), i32, i32, i32, i32, dbl, dbl, i32, i64,
                                                      C.c_uint64, pp]),
        "aps_debug_tc_slots": (i32, [vp, i64, i64]),
        "aps_debug_pair_screen": (i32, [vp, vp, i64, vp, i64, i32, vp, vp, i32]),
        "aps_debug_tc_scores": (i32, [vp, vp, i64, vp, i64, i32, i32, vp, vp, vp]),
        "aps_debug_tc_candidates": (i32, [vp, vp, i64, vp, i64, i32, i32, i32, i64, i64, i64, i64, vp, i64, vp, vp, vp,
                                          vp, vp, vp, vp, vp]),
        "aps_debug_tc_candidates_k": (i32, [vp, vp, i64, vp, i64, i32, i32, i32, i64, i64, i64, i64, vp, i64, vp, vp, vp,
                                            vp, vp, vp, vp, vp, i32]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)  # AttributeError here == the library does not export a declared symbol
        fn.restype, fn.argtypes = res, args
    L._aps_symbols = sorted(sig)
    _lib = L
    return L


def check(rc: int):
    if rc != 0:
        L = lib()
        raise ApsError(rc, L.aps_error_id().decode(), L.aps_last_error().decode())


class Context:
    """One per (process, GPU).  Creation fails loudly when there is no CUDA device."""

    def __init__(self, device: int = 0, stream: int | None = None):
        L = lib()
        h = C.c_void_p()
        check(L.aps_ctx_create(int(device), C.byref(h)))
        self._h = h
        self.device = device
        if stream is not None:
            check(L.aps_ctx_set_stream(self._h, C.c_void_p(stream)))

    @property
    def handle(self):
        return self._h

    def set_float_engine(self, engine: int):
        check(lib().aps_ctx_set_float_engine(self._h, int(engine)))

    def set_pairwise_epilogue(self, mode: int):
        """-1 = auto (default), 0 = streaming top-4, 1 = branch-free segment selection (see include/apsmatch.h)."""
        check(lib().aps_ctx_set_pairwise_epilogue(self._h, int(mode)))

    def set_pairwise_screen(self, on=True):
        """Stage 1 of the batched pairwise path (fp16 tensor screen, see include/apsmatch.h); on by default."""
        check(lib().aps_ctx_set_pairwise_screen(self._h, int(bool(on))))

    def pairwise_stats(self):
        a = (C.c_int64 * 4)()
        check(lib().aps_ctx_pairwise_stats(self._h, a))
        return {"pairs_screened": a[0], "pairs_to_exact": a[1], "entries_screened": a[2]}

    def enable_timing(self, on=True):
        check(lib().aps_ctx_enable_timing(self._h, int(bool(on))))

    def tc_time(self):
        """(summed tcgen05-kernel milliseconds, launches) since the last call; synchronises."""
        ms, n = C.c_double(0), C.c_int64(0)
        check(lib().aps_ctx_tc_time(self._h, C.byref(ms), C.byref(n)))
        return ms.value, n.value

    def synchronize(self):
        check(lib().aps_ctx_synchronize(self._h))

    def last_stats(self):
        a = (C.c_int64 * 4)()
        check(lib().aps_ctx_last_stats(self._h, a))
        return {"rows": a[0], "fallback_rows": a[1], "engine": {0: "none", 1: "exact", 2: "tcgen05"}.get(a[2], a[2]),
                "bf16_exact_operands": bool(a[3])}

    def first_pass_unproven(self):
        """Rows the first completeness proof of the last float search left to the second tensor pass."""
        return int(lib().aps_ctx_first_pass_unproven(self._h))

    def close(self):
        if getattr(self, "_h", None):
            if getattr(self, "_owner", None) is None:   # a device group's member context is released with the group
                lib().aps_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_default_ctx = {}


def default_context(device: int = 0) -> Context:
    if device not in _default_ctx:
        _default_ctx[device] = Context(device)
    return _default_ctx[device]


class DeviceGroup:
    """Several GPUs driven from this process (aps_group, include/apsmatch.h): the one-call global and pairwise entries
    spread over the members and return lists bit-identical to a single Context's.  `devices` are CUDA ordinals."""

    def __init__(self, devices, shared_members: int = 0):
        """shared_members > 0 (tests): that many members, all on the single device devices[0]
        (aps_debug_group_create_shared)."""
        L = lib()
        devs = [int(d) for d in devices]
        h = C.c_void_p()
        if shared_members:
            devs = devs[:1] * int(shared_members)
            check(L.aps_debug_group_create_shared(devs[0] if devs else 0, int(shared_members), C.byref(h)))
        else:
            arr = (C.c_int * max(len(devs), 1))(*devs)
            check(L.aps_group_create(arr, len(devs), C.byref(h)))
        self._h = h
        self.devices = tuple(devs)
        self._members = []
        for i in range(len(devs)):
            m = Context.__new__(Context)
            m._h, m.device, m._owner = C.c_void_p(L.aps_group_ctx(h, i)), devs[i], self
            self._members.append(m)

    @property
    def handle(self):
        return self._h

    def __len__(self):
        return len(self.devices)

    def ctx(self, i: int) -> Context:
        """Member i's context: its knobs and the statistics of its share of the last call."""
        return self._members[i]

    def stage_times(self, i: int):
        """Member i's device milliseconds of the last multi-member call: upload, exchange, search, finish."""
        a = (C.c_double * 4)()
        check(lib().aps_group_stage_times(self._h, int(i), a))
        return {"upload": a[0], "exchange": a[1], "search": a[2], "finish": a[3]}

    def close(self):
        if getattr(self, "_h", None):
            for m in self._members:
                m._h = None
            lib().aps_group_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_default_group = {}


def default_group(devices) -> DeviceGroup:
    """One cached group per device list (in order), like default_context."""
    key = tuple(int(d) for d in devices)
    if key not in _default_group:
        _default_group[key] = DeviceGroup(key)
    return _default_group[key]
