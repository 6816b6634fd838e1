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
  for (int i = 3; i < nrhs; ++i)
    if (!mxIsDouble(prhs[i]) || mxGetNumberOfElements(prhs[i]) != 1)
      mexErrMsgIdAndTxt("apsmatch:args", "k, ratioThr, useBF, m, maxDistance, confidence, maxIter, seed and mutual "
                                         "must be double scalars");
  aps_mex_image_sets S;
  aps_mex_collect_image_sets(prhs[0], prhs[1], prhs[2], S);
  const int B = (int)S.ns.size();
  aps_image_matches* r = nullptr;
  const uint64_t seed = nrhs > 10 ? (uint64_t)mxGetScalar(prhs[10]) : 0;
  const int mutual = nrhs > 11 ? (int)mxGetScalar(prhs[11]) : 0;
  if (B > 0 && aps_global_image_matching_sets(aps_mex_ctx(), B, S.ns.data(), S.ptrs.data(), S.counts.data(), S.D,
                                              S.dtype < 0 ? APS_F32 : S.dtype, APS_COL_MAJOR,
                                              (int)mxGetScalar(prhs[3]), mxGetScalar(prhs[4]),
                                              (int)mxGetScalar(prhs[5]), mutual, S.kp.data(),
                                              (int)mxGetScalar(prhs[6]), mxGetScalar(prhs[7]), mxGetScalar(prhs[8]),
                                              (int)mxGetScalar(prhs[9]), seed, nlhs > 3, &r) != APS_OK)
    aps_mex_fail("apsmatch:args");
  aps_mex_image_matches_outputs(nlhs, plhs, S.ns, r);
  if (nlhs > 3) {
    plhs[3] = mxCreateCellMatrix(1, (mwSize)B);
    for (int b = 0; b < B; ++b) mxSetCell(plhs[3], b, aps_mex_cells(aps_image_matches_list(r, b), S.ns[b], false));
  }
  aps_image_matches_free(r);
}
