// aps_imageMatching_mex.cpp -- the stage after featureMatching/ in one device round trip:
//   [allMatches, numMatches, tforms] = aps_imageMatching_mex(keypoints, matchesAll, mBrownLowe, maxDistance,
//                                                            inliersConfidence, maxIter [, seed])
// = top-m partner selection (PP/imageMatching/imageMatching.m:75-100), the parfor over candidate pairs with
// refineMatch + estimateTransformationRANSAC ('projective', custom 'ransac' branch; :121-156, :224-246) and the
// acceptance rule ni > 8 + 0.3 nf.  Called by the drop-in matlab/imageMatching.m.
//   keypoints  : 1 x n (or n x 1) cell of [Ni x 2] double
//   matchesAll : n x n cell, {i,j} (i<j) = [M x 2] double 1-based index pairs (empty elsewhere)
// Outputs as in imageMatching.m:62-64,159-166: allMatches = cell(n), numMatches = zeros(n), tforms = cell(n,n) with
// tforms{i,j} = model (3x3, maps image j keypoints to image i), tforms{j,i} = inv(model).
#include "aps_mex_common.h"

void mexFunction(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
  if (nrhs < 6) mexErrMsgIdAndTxt("apsmatch:args", "usage: aps_imageMatching_mex(keypoints, matchesAll, m, maxDistance, confidence, maxIter[, seed])");
  const mxArray *kpc = prhs[0], *mc = prhs[1];
  if (!mxIsCell(kpc) || !mxIsCell(mc)) mexErrMsgIdAndTxt("apsmatch:args", "keypoints and matchesAll must be cell arrays");
  const int n = (int)mxGetM(mc);
  if ((int)mxGetN(mc) != n) mexErrMsgIdAndTxt("imageMatching:InvalidMatchesAllSize", "matchesAll must be an n-by-n cell array.");
  if ((int)mxGetNumberOfElements(kpc) != n)
    mexErrMsgIdAndTxt("imageMatching:InvalidKeypointsLength", "keypoints must contain n elements (one per image).");
  std::vector<int64_t> off(1, 0), pair_ptr, counts;
  std::vector<double> kp;
  std::vector<uint32_t> rows;
  aps_mex_pool_keypoints(kpc, n, 0, kp, off);
  aps_mex_match_csr(mc, n, 0, pair_ptr, rows, counts);
  plhs[0] = mxCreateCellMatrix((mwSize)n, (mwSize)n);
  mxArray* numM = mxCreateDoubleMatrix((mwSize)n, (mwSize)n, mxREAL);
  mxArray* tf = mxCreateCellMatrix((mwSize)n, (mwSize)n);
  if (nlhs > 1) plhs[1] = numM;
  if (nlhs > 2) plhs[2] = tf;
  if (n == 0) return;
  std::vector<uint8_t> cand((size_t)n * n);
  std::vector<int64_t> lin((size_t)n * n + 1);
  int64_t np = 0;
  if (aps_select_partners(aps_mex_ctx(), counts.data(), n, (int)mxGetScalar(prhs[2]), cand.data(), lin.data(), &np) != APS_OK)
    aps_mex_fail("apsmatch:args");
  if (np == 0) return;  // imageMatching.m:102-104
  int64_t total = 0;
  for (int64_t p = 0; p < np; ++p) total += pair_ptr[lin[p] + 1] - pair_ptr[lin[p]];
  const int max_iter = (int)mxGetScalar(prhs[5]);
  const uint64_t seed = nrhs > 6 ? (uint64_t)mxGetScalar(prhs[6]) : 0;
  std::vector<int64_t> ptr((size_t)np + 1);
  std::vector<double> models((size_t)np * 9), minv((size_t)np * 9);
  std::vector<uint8_t> inl((size_t)(total > 0 ? total : 1)), acc((size_t)np);
  std::vector<int32_t> ni((size_t)np), used((size_t)np);
  if (aps_image_matching(aps_mex_ctx(), n, pair_ptr.data(), rows.data(), kp.data(), off.data(), lin.data(), np,
                         mxGetScalar(prhs[3]), mxGetScalar(prhs[4]), max_iter, nullptr, 2 * (int64_t)max_iter, seed,
                         ptr.data(), models.data(), minv.data(), inl.data(), ni.data(), acc.data(), used.data()) != APS_OK)
    aps_mex_fail("apsmatch:args");
  aps_mex_put_matches(n, pair_ptr.data(), rows.data(), lin.data(), 0, np, ptr.data(), models.data(), minv.data(),
                      inl.data(), ni.data(), acc.data(), plhs[0], mxGetPr(numM), tf);
}
