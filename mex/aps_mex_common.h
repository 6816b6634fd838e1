// aps_mex_common.h -- shared glue of the MEX gateways: one lazily created GPU context per MATLAB
// process (or parfor worker), released at mexAtExit, and status -> mexErrMsgIdAndTxt mapping that keeps
// the reference's error identifiers (PP/mex/flann_knn.cpp:94-95,126-177,202; nearest2Hamming...MEX.cpp:17-28).
// The gateways only marshal mxArrays into the C ABI of include/apsmatch.h: column-major pointers go
// through unchanged (APS_COL_MAJOR), so the host-side transposes of flann_knn.cpp:99-116 disappear.
#pragma once
#include <cstdint>
#include <string>
#include <vector>

#include "../include/apsmatch.h"
#include "mex.h"

static aps_ctx* g_aps_ctx = nullptr;
static aps_group* g_aps_group = nullptr;     // device group of the last multi-GPU call (one per process)
static std::vector<int> g_aps_group_devices;  // its CUDA ordinals
static bool g_aps_atexit = false;
static void aps_mex_cleanup(void) {
  if (g_aps_ctx) aps_ctx_destroy(g_aps_ctx);
  g_aps_ctx = nullptr;
  if (g_aps_group) aps_group_destroy(g_aps_group);
  g_aps_group = nullptr;
  g_aps_group_devices.clear();
}
static inline void aps_mex_register_cleanup(void) {
  if (!g_aps_atexit) mexAtExit(aps_mex_cleanup);
  g_aps_atexit = true;
}
static inline void aps_mex_fail(const char* fallback_id) {
  const char* id = aps_error_id();
  mexErrMsgIdAndTxt((id && id[0]) ? id : fallback_id, "%s", aps_last_error());
}
static inline aps_ctx* aps_mex_ctx(void) {
  if (!g_aps_ctx) {
    if (aps_ctx_create(0, &g_aps_ctx) != APS_OK) aps_mex_fail("apsmatch:nogpu");  // no CPU fallback
    aps_mex_register_cleanup();
  }
  return g_aps_ctx;
}
// Optional trailing `gpus` argument of the batched gateway: 1-based GPU indices (MATLAB's gpuDevice numbering), a
// real double vector of distinct positive integers; [] or absent = the default device.  Returns 0-based ordinals.
// Checked before any device is touched.
static inline std::vector<int> aps_mex_gpus(const mxArray* a) {
  std::vector<int> devs;
  if (!a || mxIsEmpty(a)) return devs;
  if (!mxIsDouble(a) || mxIsComplex(a) || mxGetNumberOfDimensions(a) != 2 || (mxGetM(a) != 1 && mxGetN(a) != 1))
    mexErrMsgIdAndTxt("apsmatch:args", "gpus must be a real double vector of GPU indices (1-based, as gpuDevice)");
  const double* v = mxGetPr(a);
  for (size_t i = 0; i < mxGetNumberOfElements(a); ++i) {
    if (!(v[i] >= 1.0 && v[i] <= 65536.0) || v[i] != (double)(int)v[i])
      mexErrMsgIdAndTxt("apsmatch:args", "gpus(%d) = %g is not a positive integer GPU index", (int)i + 1, v[i]);
    for (size_t j = 0; j < i; ++j)
      if (v[j] == v[i]) mexErrMsgIdAndTxt("apsmatch:args", "GPU %d is listed twice in gpus", (int)v[i]);
    devs.push_back((int)v[i] - 1);
  }
  return devs;
}
// One aps_group per process for the last device list used; a different list replaces it.
static inline aps_group* aps_mex_group(const std::vector<int>& devs) {
  if (g_aps_group && devs == g_aps_group_devices) return g_aps_group;
  if (g_aps_group) aps_group_destroy(g_aps_group);
  g_aps_group = nullptr;
  g_aps_group_devices.clear();
  const int rc = aps_group_create(devs.data(), (int)devs.size(), &g_aps_group);
  if (rc != APS_OK) aps_mex_fail(rc == APS_ERR_ARGS ? "apsmatch:args" : "apsmatch:nogpu");  // e.g. a GPU that does not exist
  g_aps_group_devices = devs;
  aps_mex_register_cleanup();
  return g_aps_group;
}
// allDescriptors{i}: numeric matrix, or a binaryFeatures object (its .Features, featureMatchingGlobal.m:56-75).
// *is_binary: the element is a binaryFeatures OBJECT -- the reference decides "binary" by class alone (:56); a plain
// uint8 matrix is cast to single, L2-normalised and searched with float L2 there (:76-84).
static inline const mxArray* aps_mex_features(const mxArray* cell_elem, bool* is_binary = nullptr) {
  if (is_binary) *is_binary = false;
  if (!cell_elem) return nullptr;
  if (mxIsClass(cell_elem, "binaryFeatures")) {
    if (is_binary) *is_binary = true;
    return mxGetProperty(cell_elem, 0, "Features");
  }
  return cell_elem;
}
template <class T>
static inline const void* aps_mex_to_single(const mxArray* f, std::vector<std::vector<float>>& converted) {
  const T* s = (const T*)mxGetData(f);
  converted.emplace_back(s, s + mxGetNumberOfElements(f));  // single(allDesc), featureMatchingGlobal.m:81
  return converted.back().data();
}
// Collects the cell array into pointer / count vectors; returns dtype (APS_F32 / APS_U8) and D.
// Binary (APS_U8, Hamming) iff the first non-empty element is a binaryFeatures object (featureMatchingGlobal.m:56);
// every other numeric class -- plain uint8 included -- is converted to single (:76-81).
static inline void aps_mex_collect(const mxArray* cellArr, int n, std::vector<const void*>& ptrs,
                                   std::vector<int64_t>& counts, int& dtype, int& D,
                                   std::vector<std::vector<float>>& converted) {
  ptrs.assign(n, nullptr);
  counts.assign(n, 0);
  converted.reserve((size_t)n);  // pointers into `converted` must stay valid
  dtype = -1;
  D = 0;
  for (int i = 0; i < n; ++i) {
    bool isbin = false;
    const mxArray* f = (mwSize)i < mxGetNumberOfElements(cellArr) ? aps_mex_features(mxGetCell(cellArr, i), &isbin) : nullptr;
    if (!f || mxIsEmpty(f)) continue;
    if (mxGetNumberOfDimensions(f) != 2 || mxIsComplex(f))
      mexErrMsgIdAndTxt("flann_knn:type", "descriptors must be real 2D matrices");
    if (isbin && !mxIsUint8(f)) mexErrMsgIdAndTxt("flann_knn:type", "binaryFeatures.Features must be uint8");
    if (!isbin && !mxIsNumeric(f) && !mxIsLogical(f))
      mexErrMsgIdAndTxt("flann_knn:type", "Descriptors must be single (float) or uint8 (binary)");
    const int dt = isbin ? APS_U8 : APS_F32;
    if (dtype < 0) { dtype = dt; D = (int)mxGetN(f); }
    if (dt != dtype) mexErrMsgIdAndTxt("flann_knn:type", "all descriptor matrices must have the same class");
    if ((int)mxGetN(f) != D) mexErrMsgIdAndTxt("flann_knn:dim", "all descriptor matrices must have the same width");
    counts[i] = (int64_t)mxGetM(f);
    if (isbin || mxIsSingle(f)) ptrs[i] = mxGetData(f);
    else if (mxIsDouble(f)) ptrs[i] = aps_mex_to_single<double>(f, converted);
    else if (mxIsUint8(f) || mxIsLogical(f)) ptrs[i] = aps_mex_to_single<uint8_t>(f, converted);
    else if (mxIsClass(f, "int8")) ptrs[i] = aps_mex_to_single<int8_t>(f, converted);
    else if (mxIsClass(f, "uint16")) ptrs[i] = aps_mex_to_single<uint16_t>(f, converted);
    else if (mxIsClass(f, "int16")) ptrs[i] = aps_mex_to_single<int16_t>(f, converted);
    else if (mxIsClass(f, "uint32")) ptrs[i] = aps_mex_to_single<uint32_t>(f, converted);
    else if (mxIsClass(f, "int32")) ptrs[i] = aps_mex_to_single<int32_t>(f, converted);
    else mexErrMsgIdAndTxt("flann_knn:type", "unsupported descriptor class");
  }
}
// CSR match list -> n x n cell of [M x 2] double (featureMatchingGlobal.m:155-159; untouched cells stay [])
static inline mxArray* aps_mex_cells(const aps_matchlist* ml, int n, bool fill_upper_with_0x2) {
  mxArray* out = mxCreateCellMatrix((mwSize)n, (mwSize)n);
  const int64_t* pp = aps_matchlist_pair_ptr(ml);
  const uint32_t* rows = aps_matchlist_rows(ml);
  for (int j = 0; j < n; ++j)
    for (int i = 0; i < j; ++i) {
      const int64_t c = i + (int64_t)j * n, a = pp[c], b = pp[c + 1];
      if (b == a && !fill_upper_with_0x2) continue;
      mxArray* m = mxCreateDoubleMatrix((mwSize)(b - a), 2, mxREAL);
      double* d = mxGetPr(m);
      for (int64_t r = a; r < b; ++r) {
        d[r - a] = (double)rows[2 * r];
        d[(r - a) + (b - a)] = (double)rows[2 * r + 1];
      }
      mxSetCell(out, (mwIndex)c, m);
    }
  return out;
}
