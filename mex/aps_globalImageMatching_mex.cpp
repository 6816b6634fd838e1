// aps_globalImageMatching_mex.cpp -- featureMatchingGlobal followed by imageMatching, in one call:
//   [allMatchesSets, numMatchesSets, tformsSets, matchesSets] = aps_globalImageMatching_mex(descSets, numImgs,
//       keypointsSets, k, ratioThr, useBF, m, maxDistance, confidence, maxIter[, seed[, mutual]])
// descSets{b} is what aps_featureMatching_mex('global', ...) takes for set b (1 x n_b cell of descriptor matrices or
// binaryFeatures), keypointsSets{b} what aps_imageMatching_mex takes (1 x n_b cell of [Ni x 2] double; image i has one
// keypoint row per descriptor row).  Outputs are 1 x B cells; element b is exactly what aps_imageMatchingSets_mex
// returns for set b when fed by aps_featureMatching_mex('globalsets', ...) with the same seed; matchesSets (asked for
// with a fourth output) is that 'globalsets' result.  The match lists stay on the GPU between the two stages
// (aps_global_image_matching_sets).  Called by the drop-ins matlab/globalImageMatching.m (one set) and
// matlab/globalImageMatchingSets.m.
#include "aps_mex_common.h"

void mexFunction(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
  if (nrhs < 10)
    mexErrMsgIdAndTxt("apsmatch:args", "usage: aps_globalImageMatching_mex(descSets, numImgs, keypointsSets, k, ratioThr, "
                                       "useBF, m, maxDistance, confidence, maxIter[, seed[, mutual]])");
  const mxArray *sets = prhs[0], *nums = prhs[1], *kps = prhs[2];
  if (!mxIsCell(sets) || !mxIsCell(kps))
    mexErrMsgIdAndTxt("apsmatch:args", "descSets and keypointsSets must be cell arrays");
  const int B = (int)mxGetNumberOfElements(sets);
  if (!mxIsDouble(nums) || (int)mxGetNumberOfElements(nums) != B || (int)mxGetNumberOfElements(kps) != B)
    mexErrMsgIdAndTxt("apsmatch:args", "numImgs and keypointsSets must hold one element per descriptor set");
  for (int i = 3; i < nrhs; ++i)
    if (!mxIsDouble(prhs[i]) || mxGetNumberOfElements(prhs[i]) != 1)
      mexErrMsgIdAndTxt("apsmatch:args", "k, ratioThr, useBF, m, maxDistance, confidence, maxIter, seed and mutual "
                                         "must be double scalars");
  std::vector<int> ns((size_t)B);
  std::vector<const void*> ptrs;
  std::vector<int64_t> counts;
  std::vector<double> kp;
  std::vector<std::vector<float>> converted;
  int dtype = -1, D = 0;
  for (int b = 0; b < B; ++b) {
    const double nb = mxGetPr(nums)[b];
    const mxArray *db = mxGetCell(sets, b), *kb = mxGetCell(kps, b);
    if (!(nb >= 1 && nb == (double)(int)nb)) mexErrMsgIdAndTxt("apsmatch:args", "numImgs must hold positive integers");
    const int n = (int)nb;
    if (!db || !kb || !mxIsCell(db) || !mxIsCell(kb))
      mexErrMsgIdAndTxt("apsmatch:args", "set %d: descriptors and keypoints must be cell arrays", b + 1);
    if ((int)mxGetNumberOfElements(kb) != n)
      mexErrMsgIdAndTxt("apsmatch:args", "set %d: keypoints must contain n elements (one per image).", b + 1);
    ns[b] = n;
    std::vector<const void*> p;
    std::vector<int64_t> c;
    int dt = -1, Db = 0;
    aps_mex_collect(db, n, p, c, dt, Db, converted);
    if (dt >= 0) {
      if (dtype >= 0 && dt != dtype)
        mexErrMsgIdAndTxt("flann_knn:type", "all descriptor sets must have the same class");
      if (dtype >= 0 && Db != D) mexErrMsgIdAndTxt("flann_knn:dim", "all descriptor sets must have the same width");
      dtype = dt;
      D = Db;
    }
    for (int i = 0; i < n; ++i) {
      if (c[i] == 0) continue;  // an image without descriptors takes part in no match
      const mxArray* k = mxGetCell(kb, i);
      if (!k || !mxIsDouble(k) || mxGetN(k) != 2 || (int64_t)mxGetM(k) != c[i])
        mexErrMsgIdAndTxt("apsmatch:args", "set %d: keypoints{%d} must be [Ni x 2] double with one row per descriptor",
                          b + 1, i + 1);
      const double* d = mxGetPr(k);
      for (int64_t r = 0; r < c[i]; ++r) {
        kp.push_back(d[r]);
        kp.push_back(d[r + c[i]]);
      }
    }
    ptrs.insert(ptrs.end(), p.begin(), p.end());
    counts.insert(counts.end(), c.begin(), c.end());
  }
  mxArray* allM = mxCreateCellMatrix(1, (mwSize)B);
  mxArray* numM = mxCreateCellMatrix(1, (mwSize)B);
  mxArray* tfs = mxCreateCellMatrix(1, (mwSize)B);
  mxArray* lists = mxCreateCellMatrix(1, (mwSize)B);
  for (int b = 0; b < B; ++b) {
    mxSetCell(allM, b, mxCreateCellMatrix((mwSize)ns[b], (mwSize)ns[b]));
    mxSetCell(numM, b, mxCreateDoubleMatrix((mwSize)ns[b], (mwSize)ns[b], mxREAL));
    mxSetCell(tfs, b, mxCreateCellMatrix((mwSize)ns[b], (mwSize)ns[b]));
  }
  plhs[0] = allM;
  if (nlhs > 1) plhs[1] = numM;
  if (nlhs > 2) plhs[2] = tfs;
  if (nlhs > 3) plhs[3] = lists;
  if (B == 0) return;
  const uint64_t seed = nrhs > 10 ? (uint64_t)mxGetScalar(prhs[10]) : 0;
  const int mutual = nrhs > 11 ? (int)mxGetScalar(prhs[11]) : 0;
  aps_image_matches* r = nullptr;
  if (aps_global_image_matching_sets(aps_mex_ctx(), B, ns.data(), ptrs.data(), counts.data(), D,
                                     dtype < 0 ? APS_F32 : dtype, APS_COL_MAJOR, (int)mxGetScalar(prhs[3]),
                                     mxGetScalar(prhs[4]), (int)mxGetScalar(prhs[5]), mutual, kp.data(),
                                     (int)mxGetScalar(prhs[6]), mxGetScalar(prhs[7]), mxGetScalar(prhs[8]),
                                     (int)mxGetScalar(prhs[9]), seed, nlhs > 3, &r) != APS_OK)
    aps_mex_fail("apsmatch:args");
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
    if (nlhs > 3) mxSetCell(lists, b, aps_mex_cells(aps_image_matches_list(r, b), ns[b], false));
  }
  aps_image_matches_free(r);
}
