// aps_imageMatchingSets_mex.cpp -- aps_imageMatching_mex over B independent image sets in one device pass:
//   [allMatchesSets, numMatchesSets, tformsSets] = aps_imageMatchingSets_mex(keypointsSets, matchesAllSets, m,
//                                                                            maxDistance, confidence, maxIter[, seed])
// keypointsSets{b} / matchesAllSets{b} are what aps_imageMatching_mex takes for set b (1 x n_b cell of [Ni x 2] double,
// n_b x n_b cell of [M x 2] double 1-based index pairs).  Outputs are 1 x B cells; element b is exactly what
// aps_imageMatching_mex returns for set b with the same seed.  One top-m partner selection over every set
// (aps_select_partners_sets) and one RANSAC pass over every candidate pair (aps_image_matching_sets).  Called by the
// drop-in matlab/imageMatchingSets.m.
#include "aps_mex_common.h"

void mexFunction(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
  if (nrhs < 6)
    mexErrMsgIdAndTxt("apsmatch:args", "usage: aps_imageMatchingSets_mex(keypointsSets, matchesAllSets, m, maxDistance, "
                                       "confidence, maxIter[, seed])");
  const mxArray *kps = prhs[0], *mcs = prhs[1];
  if (!mxIsCell(kps) || !mxIsCell(mcs)) mexErrMsgIdAndTxt("apsmatch:args", "keypointsSets and matchesAllSets must be cell arrays");
  const int B = (int)mxGetNumberOfElements(mcs);
  if ((int)mxGetNumberOfElements(kps) != B)
    mexErrMsgIdAndTxt("apsmatch:args", "keypointsSets and matchesAllSets must hold one element per set");
  for (int i = 2; i < nrhs; ++i)
    if (!mxIsDouble(prhs[i]) || mxGetNumberOfElements(prhs[i]) != 1)
      mexErrMsgIdAndTxt("apsmatch:args", "m, maxDistance, confidence, maxIter and seed must be double scalars");
  std::vector<int> ns((size_t)B);
  std::vector<int64_t> off(1, 0), counts;
  std::vector<double> kp;
  std::vector<std::vector<int64_t>> pair_ptr((size_t)B);
  std::vector<std::vector<uint32_t>> rows((size_t)B);
  for (int b = 0; b < B; ++b) {
    const mxArray *kpc = mxGetCell(kps, b), *mc = mxGetCell(mcs, b);
    if (!kpc || !mc || !mxIsCell(kpc) || !mxIsCell(mc))
      mexErrMsgIdAndTxt("apsmatch:args", "set %d: keypoints and matchesAll must be cell arrays", b + 1);
    const int n = (int)mxGetM(mc);
    if ((int)mxGetN(mc) != n) mexErrMsgIdAndTxt("apsmatch:args", "set %d: matchesAll must be an n-by-n cell array.", b + 1);
    if ((int)mxGetNumberOfElements(kpc) != n)
      mexErrMsgIdAndTxt("apsmatch:args", "set %d: keypoints must contain n elements (one per image).", b + 1);
    ns[b] = n;
    aps_mex_pool_keypoints(kpc, n, b + 1, kp, off);
    aps_mex_match_csr(mc, n, b + 1, pair_ptr[b], rows[b], counts);
  }
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
  if (B == 0) return;
  int64_t cap = 0;
  for (int n : ns) cap += (int64_t)n * (n - 1) / 2;
  std::vector<uint8_t> cand(counts.size() + 1);
  std::vector<int64_t> lin((size_t)cap + 1), spp((size_t)B + 1);
  if (aps_select_partners_sets(aps_mex_ctx(), B, ns.data(), counts.data(), (int)mxGetScalar(prhs[2]), cand.data(),
                               lin.data(), spp.data()) != APS_OK)
    aps_mex_fail("apsmatch:args");
  const int64_t np = spp[B];
  if (np == 0) return;  // imageMatching.m:102-104
  std::vector<const int64_t*> pps((size_t)B);
  std::vector<const uint32_t*> rps((size_t)B);
  int64_t total = 0;
  for (int b = 0; b < B; ++b) {
    pps[b] = pair_ptr[b].data();
    rps[b] = rows[b].data();
    for (int64_t p = spp[b]; p < spp[b + 1]; ++p) total += pair_ptr[b][lin[p] + 1] - pair_ptr[b][lin[p]];
  }
  const int max_iter = (int)mxGetScalar(prhs[5]);
  const uint64_t seed = nrhs > 6 ? (uint64_t)mxGetScalar(prhs[6]) : 0;
  std::vector<int64_t> ptr((size_t)np + 1);
  std::vector<double> models((size_t)np * 9), minv((size_t)np * 9);
  std::vector<uint8_t> inl((size_t)(total > 0 ? total : 1)), acc((size_t)np);
  std::vector<int32_t> ni((size_t)np), used((size_t)np);
  if (aps_image_matching_sets(aps_mex_ctx(), B, ns.data(), pps.data(), rps.data(), kp.data(), off.data(), spp.data(),
                              lin.data(), mxGetScalar(prhs[3]), mxGetScalar(prhs[4]), max_iter, nullptr,
                              2 * (int64_t)max_iter, seed, ptr.data(), models.data(), minv.data(), inl.data(), ni.data(),
                              acc.data(), used.data()) != APS_OK)
    aps_mex_fail("apsmatch:args");
  for (int b = 0; b < B; ++b)
    aps_mex_put_matches(ns[b], pair_ptr[b].data(), rows[b].data(), lin.data(), spp[b], spp[b + 1], ptr.data(),
                        models.data(), minv.data(), inl.data(), ni.data(), acc.data(), mxGetCell(allM, b),
                        mxGetPr(mxGetCell(numM, b)), mxGetCell(tfs, b));
}
