// aps_pairwiseImageMatching_mex.cpp -- featureMatchingPairwise followed by imageMatching, in one call:
//   [allMatchesSets, numMatchesSets, tformsSets, matchesSets] = aps_pairwiseImageMatching_mex(descSets, numImgs,
//       keypointsSets, matchThreshold, maxRatio, method, m, maxDistance, confidence, maxIter[, seed])
// descSets, numImgs and keypointsSets as aps_globalImageMatching_mex takes them; matchThreshold / maxRatio / method as
// aps_featureMatching_mex('pairwisesets', ...) takes them (aps_method; subset 12000 and subset seed 0, as there).
// Outputs are 1 x B cells; element b is exactly what aps_imageMatchingSets_mex returns for set b when fed by
// aps_featureMatching_mex('pairwisesets', ...) with the same seed; matchesSets (asked for with a fourth output) is that
// 'pairwisesets' result.  The match lists stay on the GPU between the two stages (aps_pairwise_image_matching_sets).
// Called by the drop-ins matlab/pairwiseImageMatching.m (one set) and matlab/pairwiseImageMatchingSets.m.
#include "aps_mex_common.h"

void mexFunction(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
  if (nrhs < 10)
    mexErrMsgIdAndTxt("apsmatch:args", "usage: aps_pairwiseImageMatching_mex(descSets, numImgs, keypointsSets, "
                                       "matchThreshold, maxRatio, method, m, maxDistance, confidence, maxIter[, seed])");
  for (int i = 3; i < nrhs; ++i)
    if (!mxIsDouble(prhs[i]) || mxGetNumberOfElements(prhs[i]) != 1)
      mexErrMsgIdAndTxt("apsmatch:args", "matchThreshold, maxRatio, method, m, maxDistance, confidence, maxIter and "
                                         "seed must be double scalars");
  aps_mex_image_sets S;
  aps_mex_collect_image_sets(prhs[0], prhs[1], prhs[2], S);
  const int B = (int)S.ns.size();
  aps_image_matches* r = nullptr;
  const uint64_t seed = nrhs > 10 ? (uint64_t)mxGetScalar(prhs[10]) : 0;
  if (B > 0 && aps_pairwise_image_matching_sets(aps_mex_ctx(), B, S.ns.data(), S.ptrs.data(), S.counts.data(), S.D,
                                                S.dtype < 0 ? APS_F32 : S.dtype, APS_COL_MAJOR, mxGetScalar(prhs[3]),
                                                mxGetScalar(prhs[4]), (int)mxGetScalar(prhs[5]), 12000, 0,
                                                S.kp.data(), (int)mxGetScalar(prhs[6]), mxGetScalar(prhs[7]),
                                                mxGetScalar(prhs[8]), (int)mxGetScalar(prhs[9]), seed, nlhs > 3,
                                                &r) != APS_OK)
    aps_mex_fail("apsmatch:args");
  aps_mex_image_matches_outputs(nlhs, plhs, S.ns, r);
  if (nlhs > 3) {  // as 'pairwisesets': every upper cell of a set with descriptors filled, [] for a set without
    plhs[3] = mxCreateCellMatrix(1, (mwSize)B);
    for (int b = 0; b < B; ++b)
      mxSetCell(plhs[3], b, S.empty[b] ? mxCreateCellMatrix((mwSize)S.ns[b], (mwSize)S.ns[b])
                                       : aps_mex_cells(aps_image_matches_list(r, b), S.ns[b], true));
  }
  aps_image_matches_free(r);
}
