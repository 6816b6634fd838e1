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
// The sets of the gateways that match and verify in one call (aps_globalImageMatching_mex, aps_pairwiseImageMatching_mex):
// descSets{b} (1 x n_b cell of descriptor matrices or binaryFeatures), numImgs(b) and keypointsSets{b} (1 x n_b cell of
// [Ni x 2] double, one row per descriptor row), checked before any device is touched.  Every image of every set one
// after another in ptrs / counts, their keypoints pooled row-major in kp; dtype < 0 when every set is empty, and
// empty[b] marks a set without descriptors.
struct aps_mex_image_sets {
  std::vector<int> ns;
  std::vector<bool> empty;
  std::vector<const void*> ptrs;
  std::vector<int64_t> counts;
  std::vector<double> kp;
  std::vector<std::vector<float>> converted;
  int dtype = -1, D = 0;
};
static inline void aps_mex_collect_image_sets(const mxArray* sets, const mxArray* nums, const mxArray* kps,
                                              aps_mex_image_sets& S) {
  if (!mxIsCell(sets) || !mxIsCell(kps))
    mexErrMsgIdAndTxt("apsmatch:args", "descSets and keypointsSets must be cell arrays");
  const int B = (int)mxGetNumberOfElements(sets);
  if (!mxIsDouble(nums) || (int)mxGetNumberOfElements(nums) != B || (int)mxGetNumberOfElements(kps) != B)
    mexErrMsgIdAndTxt("apsmatch:args", "numImgs and keypointsSets must hold one element per descriptor set");
  S.ns.assign((size_t)B, 0);
  S.empty.assign((size_t)B, true);
  for (int b = 0; b < B; ++b) {
    const double nb = mxGetPr(nums)[b];
    const mxArray *db = mxGetCell(sets, b), *kb = mxGetCell(kps, b);
    if (!(nb >= 1 && nb == (double)(int)nb)) mexErrMsgIdAndTxt("apsmatch:args", "numImgs must hold positive integers");
    const int n = (int)nb;
    if (!db || !kb || !mxIsCell(db) || !mxIsCell(kb))
      mexErrMsgIdAndTxt("apsmatch:args", "set %d: descriptors and keypoints must be cell arrays", b + 1);
    if ((int)mxGetNumberOfElements(kb) != n)
      mexErrMsgIdAndTxt("apsmatch:args", "set %d: keypoints must contain n elements (one per image).", b + 1);
    S.ns[b] = n;
    std::vector<const void*> p;
    std::vector<int64_t> c;
    int dt = -1, Db = 0;
    aps_mex_collect(db, n, p, c, dt, Db, S.converted);
    if (dt >= 0) {
      if (S.dtype >= 0 && dt != S.dtype)
        mexErrMsgIdAndTxt("flann_knn:type", "all descriptor sets must have the same class");
      if (S.dtype >= 0 && Db != S.D) mexErrMsgIdAndTxt("flann_knn:dim", "all descriptor sets must have the same width");
      S.dtype = dt;
      S.D = Db;
      S.empty[b] = false;
    }
    for (int i = 0; i < n; ++i) {
      if (c[i] == 0) continue;  // an image without descriptors takes part in no match
      const mxArray* k = mxGetCell(kb, i);
      if (!k || !mxIsDouble(k) || mxGetN(k) != 2 || (int64_t)mxGetM(k) != c[i])
        mexErrMsgIdAndTxt("apsmatch:args", "set %d: keypoints{%d} must be [Ni x 2] double with one row per descriptor",
                          b + 1, i + 1);
      const double* d = mxGetPr(k);
      for (int64_t r = 0; r < c[i]; ++r) {
        S.kp.push_back(d[r]);
        S.kp.push_back(d[r + c[i]]);
      }
    }
    S.ptrs.insert(S.ptrs.end(), p.begin(), p.end());
    S.counts.insert(S.counts.end(), c.begin(), c.end());
  }
}
// The 1 x B outputs allMatchesSets, numMatchesSets, tformsSets (imageMatching.m:148-166) of an aps_image_matches
// result r (NULL: no set) for the sets ns: allMatches{c} = the accepted pair's inlier rows, numMatches(c) = n_inliers,
// tforms{i,j} = model (maps image j to image i), tforms{j,i} = its inverse.
static inline void aps_mex_image_matches_outputs(int nlhs, mxArray* plhs[], const std::vector<int>& ns,
                                                 const aps_image_matches* r) {
  const int B = (int)ns.size();
  mxArray* allM = mxCreateCellMatrix(1, (mwSize)B);
  mxArray* numM = mxCreateCellMatrix(1, (mwSize)B);
  mxArray* tfs = mxCreateCellMatrix(1, (mwSize)B);
  for (int b = 0; b < B; ++b) {
    mxSetCell(allM, b, mxCreateCellMatrix((mwSize)ns[b], (mwSize)ns[b]));
    mxSetCell(numM, b, mxCreateDoubleMatrix((mwSize)ns[b], (mwSize)ns[b], mxREAL));
    mxSetCell(tfs, b, mxCreateCellMatrix((mwSize)ns[b], (mwSize)ns[b]));
  }
  plhs[0] = allM;
  if (nlhs > 1) plhs[1] = numM;
  if (nlhs > 2) plhs[2] = tfs;
  if (!r) return;
  const int64_t* spp = aps_image_matches_set_pair_ptr(r);
  const int64_t* lin = aps_image_matches_pairs_lin(r);
  const int64_t* mp = aps_image_matches_match_ptr(r);
  const uint32_t* rows = aps_image_matches_match_rows(r);
  const double* models = aps_image_matches_models(r);
  const double* minv = aps_image_matches_models_inv(r);
  const int32_t* ni = aps_image_matches_n_inliers(r);
  const uint8_t* acc = aps_image_matches_accepted(r);
  for (int b = 0; b < B; ++b) {
    const int64_t n = ns[b];
    mxArray *am = mxGetCell(allM, b), *tf = mxGetCell(tfs, b);
    double* nm = mxGetPr(mxGetCell(numM, b));
    for (int64_t p = spp[b]; p < spp[b + 1]; ++p) {  // imageMatching.m:148-166
      if (!acc[p]) continue;
      const int64_t c = lin[p], i = c % n, j = c / n, m = mp[p + 1] - mp[p];
      mxArray* a = mxCreateDoubleMatrix((mwSize)m, 2, mxREAL);
      for (int64_t q = 0; q < m; ++q) {
        mxGetPr(a)[q] = (double)rows[2 * (mp[p] + q)];
        mxGetPr(a)[q + m] = (double)rows[2 * (mp[p] + q) + 1];
      }
      mxSetCell(am, (mwIndex)c, a);
      nm[c] = (double)ni[p];
      mxArray *t1 = mxCreateDoubleMatrix(3, 3, mxREAL), *t2 = mxCreateDoubleMatrix(3, 3, mxREAL);
      for (int rr = 0; rr < 3; ++rr)
        for (int cc = 0; cc < 3; ++cc) {  // row-major -> MATLAB column-major
          mxGetPr(t1)[rr + 3 * cc] = models[9 * p + 3 * rr + cc];
          mxGetPr(t2)[rr + 3 * cc] = minv[9 * p + 3 * rr + cc];
        }
      mxSetCell(tf, (mwIndex)(i + j * n), t1);
      mxSetCell(tf, (mwIndex)(j + i * n), t2);
    }
  }
}
// "" or " (set b)" after a gateway message: the sets gateway names the set (1-based), the single-set one does not
static inline std::string aps_mex_in_set(int set) {
  return set > 0 ? " (set " + std::to_string(set) + ")" : std::string();
}
// keypoints{i} (1 x n or n x 1 cell of [Ni x 2] double) appended to the pooled row-major [F x 2] keypoints and their
// row offsets (off starts with {0}).  An empty [Ni x 0] element counts Ni rows with zero coordinates.
static inline void aps_mex_pool_keypoints(const mxArray* kpc, int n, int set, std::vector<double>& kp,
                                          std::vector<int64_t>& off) {
  for (int i = 0; i < n; ++i) {
    const mxArray* k = mxGetCell(kpc, i);
    if (k && !mxIsEmpty(k) && (!mxIsDouble(k) || mxGetN(k) != 2))
      mexErrMsgIdAndTxt("apsmatch:args", "keypoints{%d} must be [Ni x 2] double%s", i + 1, aps_mex_in_set(set).c_str());
    const int64_t ni = k ? (int64_t)mxGetM(k) : 0;
    const double* d = (k && !mxIsEmpty(k)) ? mxGetPr(k) : nullptr;
    for (int64_t r = 0; r < ni; ++r) {
      kp.push_back(d ? d[r] : 0.0);
      kp.push_back(d ? d[r + ni] : 0.0);
    }
    off.push_back(off.back() + ni);
  }
}
// CSR of the n x n cell's strict upper triangle (pair_ptr [n*n + 1], rows = 1-based index pairs) and the putativeCount
// of every cell (imageMatching.m:76), appended to counts
static inline void aps_mex_match_csr(const mxArray* mc, int n, int set, std::vector<int64_t>& pair_ptr,
                                     std::vector<uint32_t>& rows, std::vector<int64_t>& counts) {
  const size_t cells = (size_t)n * n;
  pair_ptr.assign(cells + 1, 0);
  for (size_t c = 0; c < cells; ++c) {
    const mxArray* e = mxGetCell(mc, c);
    counts.push_back(e ? (int64_t)mxGetM(e) : 0);
    const bool upper = (int)(c % n) < (int)(c / n);
    const bool used = upper && e && mxGetN(e) == 2 && mxGetM(e) > 0;
    if (used && !mxIsDouble(e))
      mexErrMsgIdAndTxt("apsmatch:args", "matchesAll{i,j} must be double%s", aps_mex_in_set(set).c_str());
    pair_ptr[c + 1] = pair_ptr[c] + (used ? (int64_t)mxGetM(e) : 0);
  }
  rows.resize((size_t)(2 * pair_ptr[cells]));
  for (size_t c = 0; c < cells; ++c) {
    const int64_t a = pair_ptr[c], m = pair_ptr[c + 1] - a;
    const double* d = m ? mxGetPr(mxGetCell(mc, c)) : nullptr;
    for (int64_t r = 0; r < m; ++r) {
      rows[2 * (a + r)] = (uint32_t)d[r];
      rows[2 * (a + r) + 1] = (uint32_t)d[r + m];
    }
  }
}
// One set's imageMatching outputs (imageMatching.m:148-166) from the RANSAC results of its candidate pairs [p0, p1):
// allMatches{c} = matches(inliers,:), numMatches(c) = ni, tforms{i,j} = model (maps image j to image i), tforms{j,i} =
// its inverse.  lin: cells of the set's block; pair_ptr / rows: the set's CSR; ptr: absolute offsets into inl.
static inline void aps_mex_put_matches(int64_t n, const int64_t* pair_ptr, const uint32_t* rows, const int64_t* lin,
                                       int64_t p0, int64_t p1, const int64_t* ptr, const double* models,
                                       const double* minv, const uint8_t* inl, const int32_t* ni, const uint8_t* acc,
                                       mxArray* allM, double* numM, mxArray* tf) {
  for (int64_t p = p0; p < p1; ++p) {
    if (!acc[p]) continue;
    const int64_t c = lin[p], i = c % n, j = c / n, a = pair_ptr[c], m = ptr[p + 1] - ptr[p];
    mxArray* am = mxCreateDoubleMatrix((mwSize)ni[p], 2, mxREAL);
    double* d = mxGetPr(am);
    int64_t w = 0;
    for (int64_t r = 0; r < m; ++r)
      if (inl[ptr[p] + r]) {
        d[w] = (double)rows[2 * (a + r)];
        d[w + ni[p]] = (double)rows[2 * (a + r) + 1];
        ++w;
      }
    mxSetCell(allM, (mwIndex)c, am);
    numM[c] = (double)ni[p];
    mxArray *t1 = mxCreateDoubleMatrix(3, 3, mxREAL), *t2 = mxCreateDoubleMatrix(3, 3, mxREAL);
    for (int rr = 0; rr < 3; ++rr)
      for (int cc = 0; cc < 3; ++cc) {  // row-major -> MATLAB column-major
        mxGetPr(t1)[rr + 3 * cc] = models[9 * p + 3 * rr + cc];
        mxGetPr(t2)[rr + 3 * cc] = minv[9 * p + 3 * rr + cc];
      }
    mxSetCell(tf, (mwIndex)(i + j * n), t1);
    mxSetCell(tf, (mwIndex)(j + i * n), t2);
  }
}
