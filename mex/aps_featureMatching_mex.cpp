// aps_featureMatching_mex.cpp -- batched gateway: the whole featureMatching/ stage in one device round trip.
//   matches = aps_featureMatching_mex('global',   allDescriptors, numImg, k, ratioThr, useBF [, gpus])
//   matchesSets = aps_featureMatching_mex('globalsets', {allDesc_1, ..., allDesc_B}, numImgs, k, ratioThr, useBF [, mutual])
//   matches = aps_featureMatching_mex('pairwise', allDescriptors, numImg, matchThreshold, maxRatio [, method [, gpus]])
//   [cand, IuptriIdx] = aps_featureMatching_mex('partners', matchesAll | countMatrix, m)
// Called by the drop-in matlab/featureMatchingGlobal.m / featureMatchingPairwise.m (same signatures as
// PP/featureMatching/featureMatchingGlobal.m:1 and featureMatchingPairwise.m:1), matlab/featureMatchingGlobalSets.m
// ('globalsets'), and by the two-line patch of
// PP/imageMatching/imageMatching.m:75-100 shown in INTEGRATION.md.
// gpus: optional vector of 1-based GPU indices (gpuDevice numbering).  Absent, [] or 1 = the single default context
// (device 1); any other list runs the call on a device group of those GPUs (aps_group_*, same lists).
// 'globalsets': B independent image sets in one call (aps_feature_matching_global_sets); returns a 1 x B cell whose
// element b is set b's numImgs(b) x numImgs(b) cell, exactly as 'global' returns it.  Every set uses one descriptor
// class and width.
#include "aps_mex_common.h"

static void global_sets(int nrhs, mxArray* plhs[], const mxArray* prhs[]) {
  if (nrhs < 5) mexErrMsgIdAndTxt("apsmatch:args", "globalsets: need the sets, numImgs, k and ratio threshold");
  const mxArray* sets = prhs[1];
  if (!mxIsCell(sets)) mexErrMsgIdAndTxt("apsmatch:args", "globalsets: the descriptor sets must be a cell array of cell arrays");
  const int B = (int)mxGetNumberOfElements(sets);
  const mxArray* nimg = prhs[2];
  if (!mxIsDouble(nimg) || mxIsComplex(nimg) || (int)mxGetNumberOfElements(nimg) != B)
    mexErrMsgIdAndTxt("apsmatch:args", "globalsets: numImgs must be a real double vector with one count per set");
  std::vector<int> set_images((size_t)B);
  std::vector<const void*> ptrs;
  std::vector<int64_t> counts;
  std::vector<std::vector<std::vector<float>>> keep((size_t)B);  // converted matrices of every set stay alive
  int dtype = -1, D = 0;
  for (int b = 0; b < B; ++b) {
    const double v = mxGetPr(nimg)[b];
    if (!(v >= 1.0 && v <= 2147483647.0) || v != (double)(int64_t)v)
      mexErrMsgIdAndTxt("apsmatch:args", "globalsets: numImgs(%d) = %g is not a positive integer", b + 1, v);
    const mxArray* cellb = mxGetCell(sets, (mwIndex)b);
    if (!cellb || !mxIsCell(cellb)) mexErrMsgIdAndTxt("apsmatch:args", "globalsets: set %d is not a cell array", b + 1);
    set_images[b] = (int)v;
    std::vector<const void*> pb;
    std::vector<int64_t> cb;
    int dt, Db;
    aps_mex_collect(cellb, set_images[b], pb, cb, dt, Db, keep[b]);
    if (dt >= 0) {  // one ABI call takes one class and one width
      if (dtype >= 0 && dt != dtype) mexErrMsgIdAndTxt("apsmatch:args", "globalsets: set %d has another descriptor class", b + 1);
      if (dtype >= 0 && Db != D) mexErrMsgIdAndTxt("apsmatch:args", "globalsets: set %d has another descriptor width", b + 1);
      dtype = dt;
      D = Db;
    }
    ptrs.insert(ptrs.end(), pb.begin(), pb.end());
    counts.insert(counts.end(), cb.begin(), cb.end());
  }
  const int mutual = nrhs > 6 ? (int)mxGetScalar(prhs[6]) : 0;
  std::vector<aps_matchlist*> ml((size_t)B, nullptr);
  if (dtype >= 0 && aps_feature_matching_global_sets(aps_mex_ctx(), B, set_images.data(), ptrs.data(), counts.data(), D,
                                                     dtype, APS_COL_MAJOR, (int)mxGetScalar(prhs[3]),
                                                     mxGetScalar(prhs[4]), nrhs > 5 ? (int)mxGetScalar(prhs[5]) : 0,
                                                     mutual, ml.data()) != APS_OK)
    aps_mex_fail("apsmatch:args");
  plhs[0] = mxCreateCellMatrix(1, (mwSize)B);
  for (int b = 0; b < B; ++b) {  // every set empty: cell(numImg) each, no GPU touched (featureMatchingGlobal.m:49-52)
    mxSetCell(plhs[0], (mwIndex)b, ml[b] ? aps_mex_cells(ml[b], set_images[b], false)
                                         : mxCreateCellMatrix((mwSize)set_images[b], (mwSize)set_images[b]));
    aps_matchlist_free(ml[b]);
  }
}

void mexFunction(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
  if (nrhs < 3 || !mxIsChar(prhs[0]))
    mexErrMsgIdAndTxt("apsmatch:args", "first argument must be 'global', 'globalsets', 'pairwise' or 'partners'");
  char* m = mxArrayToString(prhs[0]);
  const std::string mode = m ? m : "";
  if (m) mxFree(m);
  if (mode == "globalsets") {
    global_sets(nrhs, plhs, prhs);
    return;
  }
  if (mode == "partners") {
    const mxArray* in = prhs[1];
    const int n = (int)mxGetM(in);
    if ((int)mxGetN(in) != n) mexErrMsgIdAndTxt("imageMatching:InvalidMatchesAllSize", "matchesAll must be an n-by-n cell array.");
    std::vector<int64_t> counts((size_t)n * n, 0);
    for (size_t c = 0; c < counts.size(); ++c) {
      if (mxIsCell(in)) {
        const mxArray* e = mxGetCell(in, c);
        counts[c] = e ? (int64_t)mxGetM(e) : 0;  // putativeCount = cellfun(@(x) size(x,1), matchesAll), :76
      } else {
        counts[c] = (int64_t)mxGetPr(in)[c];
      }
    }
    plhs[0] = mxCreateLogicalMatrix((mwSize)n, (mwSize)n);
    std::vector<int64_t> lin(counts.size() + 1);
    int64_t np = 0;
    if (aps_select_partners(aps_mex_ctx(), counts.data(), n, (int)mxGetScalar(prhs[2]), (uint8_t*)mxGetData(plhs[0]),
                            lin.data(), &np) != APS_OK)
      aps_mex_fail("apsmatch:args");
    if (nlhs > 1) {
      plhs[1] = mxCreateDoubleMatrix((mwSize)np, 1, mxREAL);
      for (int64_t i = 0; i < np; ++i) mxGetPr(plhs[1])[i] = (double)(lin[i] + 1);  // find(): 1-based linear indices
    }
    return;
  }
  if (!mxIsCell(prhs[1])) mexErrMsgIdAndTxt("apsmatch:args", "allDescriptors must be a cell array");
  const std::vector<int> gpus = aps_mex_gpus(nrhs > 6 ? prhs[6] : nullptr);
  const bool grouped = !gpus.empty() && !(gpus.size() == 1 && gpus[0] == 0);
  const int n = (int)mxGetScalar(prhs[2]);
  std::vector<const void*> ptrs;
  std::vector<int64_t> counts;
  std::vector<std::vector<float>> converted;
  int dtype, D;
  aps_mex_collect(prhs[1], n, ptrs, counts, dtype, D, converted);
  if (dtype < 0) {  // all empty -> cell(numImg)   (featureMatchingGlobal.m:49-52)
    plhs[0] = mxCreateCellMatrix((mwSize)n, (mwSize)n);
    return;
  }
  aps_matchlist* ml = nullptr;
  int rc;
  if (mode == "global") {
    if (nrhs < 5) mexErrMsgIdAndTxt("apsmatch:args", "global: need k and ratio threshold");
    if (grouped) {
      rc = aps_group_feature_matching_global(aps_mex_group(gpus), ptrs.data(), counts.data(), n, D, dtype, APS_COL_MAJOR,
                                             (int)mxGetScalar(prhs[3]), mxGetScalar(prhs[4]), /*mutual*/ 0, &ml);
    } else {
      rc = aps_feature_matching_global(aps_mex_ctx(), ptrs.data(), counts.data(), n, D, dtype, APS_COL_MAJOR,
                                       (int)mxGetScalar(prhs[3]), mxGetScalar(prhs[4]),
                                       nrhs > 5 ? (int)mxGetScalar(prhs[5]) : 0, &ml);
    }
  } else if (mode == "pairwise") {
    if (nrhs < 5) mexErrMsgIdAndTxt("apsmatch:args", "pairwise: need MatchThreshold and MaxRatio");
    const int method = nrhs > 5 ? (int)mxGetScalar(prhs[5]) : APS_METHOD_EXHAUSTIVE;   // aps_method
    if (grouped) {
      rc = aps_group_feature_matching_pairwise(aps_mex_group(gpus), ptrs.data(), counts.data(), n, D, dtype,
                                               APS_COL_MAJOR, mxGetScalar(prhs[3]), mxGetScalar(prhs[4]), method, 12000,
                                               0, &ml);
    } else if (method == APS_METHOD_EXHAUSTIVE || dtype == APS_U8) {
      rc = aps_feature_matching_pairwise(aps_mex_ctx(), ptrs.data(), counts.data(), n, D, dtype, APS_COL_MAJOR,
                                         mxGetScalar(prhs[3]), mxGetScalar(prhs[4]), &ml);
    } else {   // 'subsetpdist2' / 'kdtree' (matchFeaturesScratch.m:142-155): staged plan with the Euclidean metric
      aps_pplan* plan = nullptr;
      rc = aps_pplan_create(aps_mex_ctx(), counts.data(), n, D, dtype, &plan);
      if (rc == APS_OK) rc = aps_pplan_set_method(plan, method, 12000, 0);
      if (rc == APS_OK) rc = aps_pplan_upload(plan, ptrs.data(), APS_COL_MAJOR);
      if (rc == APS_OK) rc = aps_pplan_prepare(plan);
      if (rc == APS_OK) rc = aps_pplan_match(plan, mxGetScalar(prhs[3]), mxGetScalar(prhs[4]), 0, 1, &ml);
      aps_pplan_destroy(plan);
    }
  } else {
    mexErrMsgIdAndTxt("apsmatch:args", "unknown mode '%s'", mode.c_str());
    return;
  }
  if (rc != APS_OK) aps_mex_fail("apsmatch:args");
  plhs[0] = aps_mex_cells(ml, n, mode == "pairwise");
  aps_matchlist_free(ml);
}
