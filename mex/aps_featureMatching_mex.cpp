// aps_featureMatching_mex.cpp -- batched gateway: the whole featureMatching/ stage in one device round trip.
//   matches = aps_featureMatching_mex('global',   allDescriptors, numImg, k, ratioThr, useBF [, gpus])
//   matchesSets = aps_featureMatching_mex('globalsets', {allDesc_1, ..., allDesc_B}, numImgs, k, ratioThr, useBF [, mutual])
//   matches = aps_featureMatching_mex('pairwise', allDescriptors, numImg, matchThreshold, maxRatio [, method [, gpus]])
//   matchesSets = aps_featureMatching_mex('pairwisesets', {allDesc_1, ..., allDesc_B}, numImgs, matchThreshold, maxRatio [, method])
//   [cand, IuptriIdx] = aps_featureMatching_mex('partners', matchesAll | countMatrix, m)
// Called by the drop-in matlab/featureMatchingGlobal.m / featureMatchingPairwise.m (same signatures as
// PP/featureMatching/featureMatchingGlobal.m:1 and featureMatchingPairwise.m:1), matlab/featureMatchingGlobalSets.m
// ('globalsets'), matlab/featureMatchingPairwiseSets.m ('pairwisesets'), and by the two-line patch of
// PP/imageMatching/imageMatching.m:75-100 shown in INTEGRATION.md.
// gpus: optional vector of 1-based GPU indices (gpuDevice numbering).  Absent, [] or 1 = the single default context
// (device 1); any other list runs the call on a device group of those GPUs (aps_group_*, same lists).
// 'globalsets': B independent image sets in one call (aps_feature_matching_global_sets); returns a 1 x B cell whose
// element b is set b's numImgs(b) x numImgs(b) cell, exactly as 'global' returns it.  'pairwisesets': the same for
// 'pairwise' (aps_feature_matching_pairwise_sets, subset 12000, seed 0).  Every set uses one descriptor class and width.
#include "aps_mex_common.h"

// The descriptor sets of 'globalsets' / 'pairwisesets' (prhs[1], counts prhs[2]), checked before any device is touched:
// every image of every set one after another in ptrs / counts; dtype < 0 when every set is empty.  set_dtype[b] < 0
// marks a set without descriptors.
struct MexSets {
  std::vector<int> set_images, set_dtype;
  std::vector<const void*> ptrs;
  std::vector<int64_t> counts;
  std::vector<std::vector<std::vector<float>>> keep;  // converted matrices of every set stay alive
  int dtype = -1, D = 0;
};
static void collect_sets(const char* verb, const char* scalars, int nrhs, const mxArray* prhs[], MexSets& S) {
  if (nrhs < 5) mexErrMsgIdAndTxt("apsmatch:args", "%s: need the sets, numImgs, %s", verb, scalars);
  const mxArray* sets = prhs[1];
  if (!mxIsCell(sets)) mexErrMsgIdAndTxt("apsmatch:args", "%s: the descriptor sets must be a cell array of cell arrays", verb);
  const int B = (int)mxGetNumberOfElements(sets);
  const mxArray* nimg = prhs[2];
  if (!mxIsDouble(nimg) || mxIsComplex(nimg) || (int)mxGetNumberOfElements(nimg) != B)
    mexErrMsgIdAndTxt("apsmatch:args", "%s: numImgs must be a real double vector with one count per set", verb);
  S.set_images.assign((size_t)B, 0);
  S.set_dtype.assign((size_t)B, -1);
  S.keep.resize((size_t)B);
  for (int b = 0; b < B; ++b) {
    const double v = mxGetPr(nimg)[b];
    if (!(v >= 1.0 && v <= 2147483647.0) || v != (double)(int64_t)v)
      mexErrMsgIdAndTxt("apsmatch:args", "%s: numImgs(%d) = %g is not a positive integer", verb, b + 1, v);
    const mxArray* cellb = mxGetCell(sets, (mwIndex)b);
    if (!cellb || !mxIsCell(cellb)) mexErrMsgIdAndTxt("apsmatch:args", "%s: set %d is not a cell array", verb, b + 1);
    S.set_images[b] = (int)v;
    std::vector<const void*> pb;
    std::vector<int64_t> cb;
    int dt, Db;
    aps_mex_collect(cellb, S.set_images[b], pb, cb, dt, Db, S.keep[b]);
    if (dt >= 0) {  // one ABI call takes one class and one width
      if (S.dtype >= 0 && dt != S.dtype) mexErrMsgIdAndTxt("apsmatch:args", "%s: set %d has another descriptor class", verb, b + 1);
      if (S.dtype >= 0 && Db != S.D) mexErrMsgIdAndTxt("apsmatch:args", "%s: set %d has another descriptor width", verb, b + 1);
      S.dtype = dt;
      S.D = Db;
    }
    S.set_dtype[b] = dt;
    S.ptrs.insert(S.ptrs.end(), pb.begin(), pb.end());
    S.counts.insert(S.counts.end(), cb.begin(), cb.end());
  }
}

// 1 x B cell of the sets' lists; a set without descriptors gets cell(numImgs(b)), as the single-set verbs return it
static void sets_output(mxArray* plhs[], const MexSets& S, std::vector<aps_matchlist*>& ml, bool pairwise) {
  const int B = (int)S.set_images.size();
  plhs[0] = mxCreateCellMatrix(1, (mwSize)B);
  for (int b = 0; b < B; ++b) {
    const int n = S.set_images[b];
    const bool listed = ml[b] && (!pairwise || S.set_dtype[b] >= 0);
    mxSetCell(plhs[0], (mwIndex)b, listed ? aps_mex_cells(ml[b], n, pairwise) : mxCreateCellMatrix((mwSize)n, (mwSize)n));
    aps_matchlist_free(ml[b]);
  }
}

static void global_sets(int nrhs, mxArray* plhs[], const mxArray* prhs[]) {
  MexSets S;
  collect_sets("globalsets", "k and ratio threshold", nrhs, prhs, S);
  const int B = (int)S.set_images.size();
  const int mutual = nrhs > 6 ? (int)mxGetScalar(prhs[6]) : 0;
  std::vector<aps_matchlist*> ml((size_t)B, nullptr);
  if (S.dtype >= 0 && aps_feature_matching_global_sets(aps_mex_ctx(), B, S.set_images.data(), S.ptrs.data(),
                                                       S.counts.data(), S.D, S.dtype, APS_COL_MAJOR,
                                                       (int)mxGetScalar(prhs[3]), mxGetScalar(prhs[4]),
                                                       nrhs > 5 ? (int)mxGetScalar(prhs[5]) : 0, mutual,
                                                       ml.data()) != APS_OK)
    aps_mex_fail("apsmatch:args");
  sets_output(plhs, S, ml, false);  // every set empty: cell(numImg) each, no GPU touched (featureMatchingGlobal.m:49-52)
}

// as 'pairwise' per set, with its subset (12000) and seed (0)
static void pairwise_sets(int nrhs, mxArray* plhs[], const mxArray* prhs[]) {
  MexSets S;
  collect_sets("pairwisesets", "MatchThreshold and MaxRatio", nrhs, prhs, S);
  const int B = (int)S.set_images.size();
  const int method = nrhs > 5 ? (int)mxGetScalar(prhs[5]) : APS_METHOD_EXHAUSTIVE;   // aps_method
  std::vector<aps_matchlist*> ml((size_t)B, nullptr);
  if (S.dtype >= 0 && aps_feature_matching_pairwise_sets(aps_mex_ctx(), B, S.set_images.data(), S.ptrs.data(),
                                                         S.counts.data(), S.D, S.dtype, APS_COL_MAJOR,
                                                         mxGetScalar(prhs[3]), mxGetScalar(prhs[4]), method, 12000, 0,
                                                         ml.data()) != APS_OK)
    aps_mex_fail("apsmatch:args");
  sets_output(plhs, S, ml, true);
}

void mexFunction(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
  if (nrhs < 3 || !mxIsChar(prhs[0]))
    mexErrMsgIdAndTxt("apsmatch:args",
                      "first argument must be 'global', 'globalsets', 'pairwise', 'pairwisesets' or 'partners'");
  char* m = mxArrayToString(prhs[0]);
  const std::string mode = m ? m : "";
  if (m) mxFree(m);
  if (mode == "globalsets") {
    global_sets(nrhs, plhs, prhs);
    return;
  }
  if (mode == "pairwisesets") {
    pairwise_sets(nrhs, plhs, prhs);
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
