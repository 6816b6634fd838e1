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
  std::vector<int64_t> off(1, 0), counts, cell0(1, 0);
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
    for (int i = 0; i < n; ++i) {  // pooled keypoints, row-major [F x 2]
      const mxArray* k = mxGetCell(kpc, i);
      if (k && !mxIsEmpty(k) && (!mxIsDouble(k) || mxGetN(k) != 2))
        mexErrMsgIdAndTxt("apsmatch:args", "set %d: keypoints{%d} must be [Ni x 2] double", b + 1, i + 1);
      const int64_t ni = k ? (int64_t)mxGetM(k) : 0;  // rows, as aps_imageMatching_mex counts them
      const double* d = (k && !mxIsEmpty(k)) ? mxGetPr(k) : nullptr;  // an [Ni x 0] array has no coordinates: zeros
      for (int64_t r = 0; r < ni; ++r) {
        kp.push_back(d ? d[r] : 0.0);
        kp.push_back(d ? d[r + ni] : 0.0);
      }
      off.push_back(off.back() + ni);
    }
    // CSR of the set's cell (strict upper triangle) + putative counts of every cell (imageMatching.m:76)
    const size_t cells = (size_t)n * n;
    std::vector<int64_t>& pp = pair_ptr[b];
    pp.assign(cells + 1, 0);
    for (size_t c = 0; c < cells; ++c) {
      const mxArray* e = mxGetCell(mc, c);
      counts.push_back(e ? (int64_t)mxGetM(e) : 0);
      const bool upper = (int)(c % n) < (int)(c / n);
      const bool used = upper && e && mxGetN(e) == 2 && mxGetM(e) > 0;
      if (used && !mxIsDouble(e)) mexErrMsgIdAndTxt("apsmatch:args", "set %d: matchesAll{i,j} must be double", b + 1);
      pp[c + 1] = pp[c] + (used ? (int64_t)mxGetM(e) : 0);
    }
    rows[b].resize((size_t)(2 * pp[cells]));
    for (size_t c = 0; c < cells; ++c) {
      const int64_t a = pp[c], m = pp[c + 1] - a;
      const double* d = m ? mxGetPr(mxGetCell(mc, c)) : nullptr;
      for (int64_t r = 0; r < m; ++r) {
        rows[b][2 * (a + r)] = (uint32_t)d[r];
        rows[b][2 * (a + r) + 1] = (uint32_t)d[r + m];
      }
    }
    cell0.push_back(cell0.back() + (int64_t)cells);
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
  std::vector<uint8_t> cand((size_t)cell0[B] + 1);
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
  for (int b = 0; b < B; ++b) {
    const int64_t n = ns[b];
    mxArray *am_b = mxGetCell(allM, b), *tf_b = mxGetCell(tfs, b);
    double* num_b = mxGetPr(mxGetCell(numM, b));
    for (int64_t p = spp[b]; p < spp[b + 1]; ++p) {
      if (!acc[p]) continue;
      const int64_t c = lin[p], i = c % n, j = c / n, a = pair_ptr[b][c], m = ptr[p + 1] - ptr[p];
      mxArray* am = mxCreateDoubleMatrix((mwSize)ni[p], 2, mxREAL);  // matches(inliers,:), :148
      double* d = mxGetPr(am);
      int64_t w = 0;
      for (int64_t r = 0; r < m; ++r)
        if (inl[ptr[p] + r]) {
          d[w] = (double)rows[b][2 * (a + r)];
          d[w + ni[p]] = (double)rows[b][2 * (a + r) + 1];
          ++w;
        }
      mxSetCell(am_b, (mwIndex)c, am);
      num_b[c] = (double)ni[p];
      mxArray *t1 = mxCreateDoubleMatrix(3, 3, mxREAL), *t2 = mxCreateDoubleMatrix(3, 3, mxREAL);
      for (int rr = 0; rr < 3; ++rr)
        for (int cc = 0; cc < 3; ++cc) {  // row-major -> MATLAB column-major
          mxGetPr(t1)[rr + 3 * cc] = models[9 * p + 3 * rr + cc];
          mxGetPr(t2)[rr + 3 * cc] = minv[9 * p + 3 * rr + cc];
        }
      mxSetCell(tf_b, (mwIndex)(i + j * n), t1);  // tforms(IuptriIdx) = tforms_ij  (:165)
      mxSetCell(tf_b, (mwIndex)(j + i * n), t2);  // tforms(IlowtriIdx) = tforms_ji (:166)
    }
  }
}
