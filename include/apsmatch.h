/*
 * apsmatch.h -- C ABI of libapsmatch.so: the B200 (sm_100a) implementation of AutoPanoStitch's
 * featureMatching/ hot path.  Plain pointers and sizes only; no CUDA, torch or MATLAB types.
 *
 * PP/ = "Procedural Program/" in preethamam/AutomaticPanoramicImageStitching-AutoPanoStitch-MATLAB.
 * Every entry point names the reference interface it replaces.  The MEX gateways in mex/ and the
 * Python host mirror in the package bind exactly these symbols (see INTEGRATION.md).
 *
 * Conventions
 *   - status: 0 = APS_OK, otherwise an APS_ERR_* code; aps_last_error() gives the message and
 *     aps_error_id() the MATLAB error identifier the reference would have raised for it.
 *   - there is NO CPU fallback: without a usable CUDA device every compute entry returns
 *     APS_ERR_NOGPU (the reference's silent canUseGPU() fallback, matchFeaturesScratch.m:575-585,
 *     is deliberately not reproduced).
 *   - `layout`: APS_COL_MAJOR is the mxGetData layout of a MATLAB [N x D] matrix (element (r,c) at
 *     r + c*N); APS_ROW_MAJOR is a C / NumPy [N][D] array.  Outputs that are matrices use the same
 *     layout as the inputs of the call.
 *   - indices returned are 1-based, exactly as the reference returns them.
 *   - host entry points (aps_*) take HOST pointers and are synchronous.  The staged plan API
 *     (aps_gplan_*) exposes the same pipeline step by step on the context's stream, with DEVICE
 *     buffers reachable for collectives (NCCL broadcast / all-gather between ranks).
 */
#ifndef APSMATCH_H
#define APSMATCH_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define APS_ABI_VERSION 1

enum aps_status {
  APS_OK = 0,
  APS_ERR_ARGS = 1,  /* flann_knn:args / hamm2nn:nrhs : bad argument count or null pointer       */
  APS_ERR_TYPE = 2,  /* flann_knn:type / hamm2nn:type : unsupported descriptor class             */
  APS_ERR_K = 3,     /* flann_knn:k                   : k <= 0 (or k > APS_MAX_K)                */
  APS_ERR_DIM = 4,   /* flann_knn:dim / hamm2nn:cols  : descriptor width mismatch                */
  APS_ERR_BF = 5,    /* flann_knn:bf                  : 'bf' requested for float descriptors     */
  APS_ERR_NOGPU = 6, /* no CUDA device / driver: the product has no CPU path                     */
  APS_ERR_CUDA = 7,  /* a CUDA call failed; message carries cudaGetErrorString                   */
  APS_ERR_ALLOC = 8,
  APS_ERR_METHOD = 9 /* unknown method string                                                    */
};

enum aps_layout { APS_COL_MAJOR = 0, APS_ROW_MAJOR = 1 };
enum aps_dtype { APS_F32 = 0, APS_U8 = 1 };

#define APS_MAX_K 32 /* neighbours per query supported by the kNN entry points; the reference accepts any k > 0
                       (PP/mex/flann_knn.cpp:154-157) and its pipeline uses input.k = 4 and 2.  k <= 12 on float
                       descriptors runs the tcgen05 search (8 candidates per list for k <= 5, 16 for 6 <= k <= 12),
                       larger k the exact CUDA-core engine; above 32: flann_knn:k */

typedef struct aps_ctx aps_ctx;             /* one per (process, GPU): device buffers, stream          */
typedef struct aps_matchlist aps_matchlist; /* CSR form of the reference's n x n `matches` cell        */
typedef struct aps_gplan aps_gplan;         /* staged global-matching pipeline (multi-GPU building block) */

/* ---- context -------------------------------------------------------------------------------
 * No function of the reference corresponds to these: the context stands in for the state a MATLAB process or
 * parfor worker holds between MEX calls (PP/main.m:41-45 opens the pool, PP/featureMatching/
 * featureMatchingPairwise.m:54-59 runs the matcher on its workers).  The gateways create one lazily per process and
 * GPU and release it with mexAtExit (mex/aps_mex_common.h).  aps_last_error / aps_error_id carry what the
 * reference passes to mexErrMsgIdAndTxt(id, msg) (PP/mex/flann_knn.cpp:94-95,126-177,202;
 * PP/mex/nearest2HammingExhaustiveMEX.cpp:17-28). */
int aps_ctx_create(int device, aps_ctx** out);
void aps_ctx_destroy(aps_ctx* ctx);
/* Use an existing cudaStream_t (e.g. torch's current stream) instead of the context's own. */
int aps_ctx_set_stream(aps_ctx* ctx, void* cuda_stream);
int aps_ctx_synchronize(aps_ctx* ctx);
const char* aps_last_error(void); /* thread-local */
const char* aps_error_id(void);   /* e.g. "flann_knn:type"; "" when no MATLAB id applies */
int aps_abi_version(void);
/* Force a search engine for float descriptors: 0 = auto (tcgen05 candidates + exact FP32 re-rank
 * when the shape allows, else exact CUDA-core search), 1 = exact CUDA-core search only,
 * 2 = tcgen05 path required (error if the shape is unsupported).  Either way k > 12 runs the exact engine. */
int aps_ctx_set_float_engine(aps_ctx* ctx, int engine);
/* Epilogue of the batched pairwise tensor pass (aps_feature_matching_pairwise*, float descriptors): 0 = streaming
 * top-4 list per (query, train image); 1 = branch-free "two best per 64-column segment" selection with two sorted
 * lists of three per query and four epilogue warps per SM sub-partition; -1 = auto [default]: 1 when the train
 * images average at most 48 tiles of 128 descriptors, else 0.  Results are identical (both feed the exact re-rank
 * and its completeness proof); only speed and the share of rows sent to the exact fallback differ. */
int aps_ctx_set_pairwise_epilogue(aps_ctx* ctx, int mode);
/* Stage 1 of the batched pairwise path (float descriptors): 1 = on [default] -- every (query row, train image) is first
 * screened on the tensor cores with fp16 operands and fp16 accumulators; image pairs in which no query row can pass
 * the ratio / threshold test of matchFeaturesScratch.m:174-178 (proven from error-bounded distance bounds) skip the
 * exact search, their cell is empty.  0 = off: every pair goes through the exact pipeline.  Results are identical.
 * aps_ctx_pairwise_stats: [0] image pairs screened, [1] pairs that went on to the exact pipeline, [2] (query row,
 * train image) entries screened, [3] reserved -- of the last aps_pplan_match / aps_feature_matching_pairwise call. */
int aps_ctx_set_pairwise_screen(aps_ctx* ctx, int mode);
int aps_ctx_pairwise_stats(aps_ctx* ctx, int64_t stats[4]);
/* Counters of the last float search on this context: [0] rows searched, [1] rows whose
 * candidate set could not be PROVEN complete and were re-searched exactly, [2] engine used
 * (1 exact, 2 tcgen05), [3] 1 if operands were exactly representable in bf16. */
int aps_ctx_last_stats(aps_ctx* ctx, int64_t stats[4]);
/* Rows the FIRST completeness proof of the last float search left unproven (they got the second, 32-candidate tensor
 * pass; aps_ctx_last_stats[1] counts what even that could not prove and the exact engine searched). */
int64_t aps_ctx_first_pass_unproven(aps_ctx* ctx);
/* Measurement hooks (bench.py): with timing enabled the float search brackets every launch of the
 * tcgen05 candidate kernel with CUDA events on the context's stream; aps_ctx_tc_time() synchronises,
 * returns the summed kernel time and launch count since the last call, and resets them.
 * aps_launch_count() = kernels launched by this library in this process so far. */
int aps_ctx_enable_timing(aps_ctx* ctx, int enable);
int aps_ctx_tc_time(aps_ctx* ctx, double* ms_total, int64_t* launches);
int64_t aps_launch_count(void);
/* Pinned host memory for callers that want asynchronous-speed copies (bench, MEX staging) -- the descriptor cells the
 * producer hands over (PP/featureMatching/getFeaturePoints.m:32-74 -> allDescriptors, PP/main.m:95-99) can be staged here. */
void* aps_host_alloc(size_t bytes);
void aps_host_free(void* p);

/* ---- flann_knn_win(train, query, k, method, trees, checks) ------------- PP/mex/flann_knn.cpp:118-253
 * idx [Fq x k] uint32 1-based, dist [Fq x k] float, ascending; missing neighbours idx 0 / +inf
 * (:216-219).  float: SQUARED L2 with FLANN's L2 functor order, EXACT search (the reference's
 * KD-tree(4)/checks=32 is approximate: results here are the exhaustive answer of the same
 * contract).  uint8: Hamming bit counts, exact for both 'bf' (:199-223) and 'flann' (:235-240,
 * LSH in the reference).  method NULL = "flann".  trees/checks are accepted and ignored.
 * Errors mirror :125-177,:201-202 (float + 'bf' -> APS_ERR_BF, k<=0 -> APS_ERR_K ...). */
int aps_flann_knn(aps_ctx* ctx, const void* train, int64_t Ft, const void* query, int64_t Fq, int D, int dtype,
                  int layout, int k, const char* method, int trees, int checks, uint32_t* idx, float* dist);

/* ---- [idx2,d1,d2] = nearest2HammingExhaustiveMEX(A,B) / ...OMPMEX(A,B) ----------------------
 * PP/mex/nearest2HammingExhaustiveMEX.cpp:16-80, PP/mex/nearest2HammingExhaustiveOMPMEX.cpp:18-83.
 * best = first index attaining the minimum, d2 = second smallest value with multiplicity,
 * N2==0 -> idx 0 / NaN / NaN, N2==1 -> d2 = 8*nb. */
int aps_nearest2_hamming(aps_ctx* ctx, const uint8_t* A, int64_t N1, const uint8_t* B, int64_t N2, int nb,
                         int layout, uint32_t* idx2, float* d1, float* d2);

/* ---- [~,idx2,d1,d2] = nearest2SSDExhaustive(A,B) --- PP/featureMatching/matchFeaturesScratch.m:322-366
 * D2 = a2 + b2' - 2*A*B' in float32 (fixed sequential summation order), first index on ties,
 * d2 = min over j != idx2, no clamp at zero; N2==1 -> d2 = +inf; N2==0 -> idx 0, +inf, +inf. */
int aps_nearest2_ssd(aps_ctx* ctx, const float* A, int64_t N1, const float* B, int64_t N2, int D, int layout,
                     uint32_t* idx2, float* d1, float* d2);

/* ---- [matches, metric] = matchFeaturesScratch(F1,F2,'Method','Exhaustive',...) ---------------
 * PP/featureMatching/matchFeaturesScratch.m:1-215 (exhaustive branches :116-126, filters :169-215).
 * dtype APS_U8 = packed binaryFeatures rows (nBits = 8*D); APS_F32 = float descriptors, L2-normalised
 * iff max|.|>2 (:105-110).  matches: caller buffer of 2*N1 uint32, interleaved (query,train) rows;
 * metric: N1 doubles.  *K receives the number of matches. */
int aps_match_features(aps_ctx* ctx, const void* F1, int64_t N1, const void* F2, int64_t N2, int D, int dtype,
                       int layout, double match_threshold, double max_ratio, int unique, uint32_t* matches,
                       double* metric, int64_t* K);

/* Same for UNPACKED binary descriptors (logical / 0-1 uint8 matrices [N x Dbits], matchFeaturesScratch.m:259-275):
 * the bits are packed MSB-first on the device (packBits, :617-646) and nBits = Dbits enters the percent metric. */
int aps_match_features_bits(aps_ctx* ctx, const uint8_t* F1, int64_t N1, const uint8_t* F2, int64_t N2, int Dbits,
                            int layout, double match_threshold, double max_ratio, int unique, uint32_t* matches,
                            double* metric, int64_t* K);

/* ---- matches = featureMatchingGlobal(input, allDescriptors, numImg) --------------------------
 * PP/featureMatching/featureMatchingGlobal.m:1-163.  desc[i] -> image i's [counts[i] x D] matrix
 * (may be NULL when counts[i]==0).  k = input.k, ratio = input.Ratiothreshold.  use_bf is accepted
 * for interface parity (binary search is exact either way). */
int aps_feature_matching_global(aps_ctx* ctx, const void* const* desc, const int64_t* counts, int n, int D,
                                int dtype, int layout, int k, double ratio, int use_bf, aps_matchlist** out);

/* Same stage for descriptors that already live on the device (the step before the path, PP/featureMatching/
 * getFeaturePoints.m:32-74 -> allDescriptors, when the extractor runs on the GPU): d_pooled = pooled ROW-major [F x D]
 * device matrix (image i = rows sum(counts[0..i)) ...), float32 or uint8.  mutual != 0 adds the opt-in cross-check
 * (aps_gplan_filter_mutual).  The match list comes back on the host like aps_feature_matching_global's. */
int aps_feature_matching_global_dev(aps_ctx* ctx, const void* d_pooled, const int64_t* counts, int n, int D, int dtype,
                                    int k, double ratio, int mutual, aps_matchlist** out);

/* featureMatchingGlobal over nsets independent image sets in one call.  Set b has set_images[b] images; desc / counts
 * list the images of all sets one after another (set 0's images first).  Every set's match list is BIT-IDENTICAL to
 * aps_feature_matching_global (mutual = 0) or to the staged plan with aps_gplan_filter_mutual (mutual != 0) on that set
 * alone: rows of one set never see rows of another.  out[b] receives set b's list (n = set_images[b]); free each with
 * aps_matchlist_free.  All sets share one D and dtype.  Argument errors carry the ids of aps_feature_matching_global
 * (flann_knn:k, flann_knn:type, flann_knn:dim); nsets < 0, a negative count or a NULL out is APS_ERR_ARGS.
 * All sets share ONE pass, whatever nsets: one normalisation, one tcgen05 unit-table search over the float sets the
 * single-set call would search on the tensor path (each 256-row block against its own set's rows) with one re-rank and
 * one set-restricted exact fallback, one set-restricted exact (float) or Hamming (binary) search over the other sets,
 * one filter, one per-set compaction (sum of n_b^2 cells) and one download -- its launches and synchronisations do not
 * depend on nsets.  nsets == 1 is exactly the single-set call. */
int aps_feature_matching_global_sets(aps_ctx* ctx, int nsets, const int* set_images, const void* const* desc,
                                     const int64_t* counts, int D, int dtype, int layout, int k, double ratio,
                                     int use_bf, int mutual, aps_matchlist** out);

/* ---- matches = featureMatchingPairwise(input, allDescriptors, numImg) ------------------------
 * PP/featureMatching/featureMatchingPairwise.m:1-63 with getMatches :103-120 on the
 * matchFeaturesScratch 'Exhaustive' branch (input.useMATLABFeatureMatch = 0), Unique = true. */
int aps_feature_matching_pairwise(aps_ctx* ctx, const void* const* desc, const int64_t* counts, int n, int D,
                                  int dtype, int layout, double match_threshold, double max_ratio,
                                  aps_matchlist** out);

/* Multi-GPU building block of the pairwise path: computes only the image pairs whose ordinal in the
 * column-major strict-upper-triangle list (featureMatchingPairwise.m:48) is congruent to pair_first modulo
 * pair_stride (one share per rank, like the reference's parfor over the same list); other cells stay empty. */
int aps_feature_matching_pairwise_shard(aps_ctx* ctx, const void* const* desc, const int64_t* counts, int n, int D,
                                        int dtype, int layout, double match_threshold, double max_ratio,
                                        int pair_first, int pair_stride, aps_matchlist** out);

/* featureMatchingPairwise over nsets independent image sets in one call.  Set b has set_images[b] images; desc / counts
 * list the images of all sets one after another (set 0's images first).  out[b] receives set b's list (n =
 * set_images[b], with metric); free each with aps_matchlist_free.  Every list is BIT-IDENTICAL in pair_ptr, rows and
 * metric to set b matched alone with the same method, subset and seed -- aps_feature_matching_pairwise for
 * APS_METHOD_EXHAUSTIVE, the staged plan with aps_pplan_set_method otherwise (aps_method; binary descriptors run the
 * exhaustive Hamming search for every method): pairs never cross a set, and an image's 'subsetpdist2' subset is keyed
 * by its index in its own set.  All sets share one D and dtype.  Argument errors carry the single-set call's statuses;
 * nsets < 0, a negative count or a NULL out is APS_ERR_ARGS, and so is a call whose pooled rows, the subset views
 * included, reach the one-plan limit of 2^31 - 512.  nsets == 0 succeeds and returns nothing; a set with fewer than two
 * non-empty images gets an all-empty list; nsets == 1 is exactly the single-set call.
 * All sets share ONE pass, whatever nsets: one upload (one transpose launch for column-major input), one K1, one train
 * view, one pair list of every set's column-major strict upper triangle, each set's pairs on the engine its single-set
 * call chooses (fp16 screen + tcgen05 + exact re-rank, or the exact engine), batches bounded by rows, not by sets, and
 * one split into the nsets lists (sum of n_b^2 cells) -- its launches and synchronisations do not depend on nsets.
 * The flag words of a view (exactness, max |x|^2, the screen's bound) are pooled over all sets: one set's values can
 * let more pairs through another set's screen and send more of its rows to the exact fallback; the lists do not change.
 * aps_ctx_last_stats and aps_ctx_pairwise_stats report sums over the call; last_stats[2] is 2 when any set ran on the
 * tensor path. */
int aps_feature_matching_pairwise_sets(aps_ctx* ctx, int nsets, const int* set_images, const void* const* desc,
                                       const int64_t* counts, int D, int dtype, int layout, double match_threshold,
                                       double max_ratio, int method, int64_t subset, uint64_t seed, aps_matchlist** out);

/* ---- match list: the n x n cell in CSR form ---------------------------------------------------
 * cell (i,j) (0-based, i<j) is linear index c = i + j*n (MATLAB's column-major cell index);
 * its rows are rows[2*pair_ptr[c] .. 2*pair_ptr[c+1]) interleaved (col1,col2) = (index into image i,
 * index into image j), 1-based -- the layout imageMatching.m:229-230 and
 * bundleAdjustmentRKf.m:430-431 consume.  metric is NULL for global lists. */
int aps_matchlist_n(const aps_matchlist* m);
int64_t aps_matchlist_total(const aps_matchlist* m);
const int64_t* aps_matchlist_pair_ptr(const aps_matchlist* m); /* n*n + 1 entries */
const uint32_t* aps_matchlist_rows(const aps_matchlist* m);    /* 2 * total entries */
const double* aps_matchlist_metric(const aps_matchlist* m);
void aps_matchlist_free(aps_matchlist* m);

/* ---- top-m image-partner selection ------------------------- PP/imageMatching/imageMatching.m:75-100
 * counts: putativeCount [n x n] column-major (counts[i + j*n] = size(matchesAll{i,j},1)), m =
 * input.mBrownLowe.  cand [n x n] column-major logical (strict upper triangle); pairs_lin (may be
 * NULL) receives find(candidatePairs) as 0-based linear indices, *npairs their number. */
int aps_select_partners(aps_ctx* ctx, const int64_t* counts, int n, int m, uint8_t* cand, int64_t* pairs_lin,
                        int64_t* npairs);
/* The same for nsets independent image sets in one call.  Set b has set_images[b] images; counts holds, for each set,
 * its n_b x n_b column-major putativeCount block at cell_off[b] = sum_{c<b} n_c^2 (the cell layout of
 * aps_feature_matching_global_sets' compaction); cand [sum n_b^2] the blocks of candidatePairs.  pairs_lin [<= sum
 * n_b (n_b - 1) / 2] receives the 0-based linear cell indices INSIDE each set's block, set-major and ascending within a
 * set (find() order); set_pair_ptr [nsets + 1] the offset of each set's pairs.  Set b's results are bit-identical to
 * aps_select_partners on set b alone.  One upload, one download and one synchronisation, whatever nsets.  nsets < 0, a
 * negative image count or a NULL argument is APS_ERR_ARGS (checked before the context). */
int aps_select_partners_sets(aps_ctx* ctx, int nsets, const int* set_images, const int64_t* counts, int m,
                             uint8_t* cand, int64_t* pairs_lin, int64_t* set_pair_ptr);

/* ---- consumer of the match lists: batched RANSAC homographies (SURVEY.md 8(f) rank 1) ---------------
 * Replaces the parfor of PP/imageMatching/imageMatching.m:121-156 with its callee
 * PP/imageMatching/estimateTransformationRANSAC.m ('projective' = PP/inputs.m:73; :94-183 loop + refit on
 * all inliers, :188-225 normalised DLT, :444-516 symmetric transfer error, :518-530 checkModel,
 * :532-572 isDegenerate).  All trials of all pairs are evaluated in parallel (one thread per trial),
 * then the reference's sequential bookkeeping (best model, adaptive trial bound) is replayed.
 *
 * Candidate pair p owns correspondences pt_ptr[p] .. pt_ptr[p+1] (pt_ptr[0] = 0) of pts1 / pts2
 * ([total x 2] ROW-major doubles): pts1 = matchedPoints1 = keypoints of image jj, pts2 = keypoints of
 * image ii (refineMatch passes (matchedPts_2, matchedPts_1), imageMatching.m:242); the model maps pts1 -> pts2.
 * Random minimal samples: `samples` [n_pairs x n_draws x 4] zero-based row indices within the pair, or NULL
 * to draw them on the device from `seed` (aps_ransac_sample_table returns exactly that table).  Loop
 * iteration d of a pair consumes draw d (valid or skipped); the loop also ends when the table is exhausted
 * (n_draws >= 2 * max_trials reproduces the reference unless more than max_trials samples are invalid).
 * max_distance / confidence / max_trials = input.maxDistance / inliersConfidence / maxIter (PP/inputs.m:68-72).
 * Outputs (caller-allocated): models, models_inv [n_pairs x 9] ROW-major 3x3 (tforms{ii,jj}, tforms{jj,ii} =
 * inv(model); NaN when nothing was found / not accepted), inliers [total] 0/1, n_inliers, accepted
 * (ni > 8 + 0.3 nf, imageMatching.m:147; pairs with nf < 4 are skipped as in :133), draws_used.
 * Double precision; per-trial arithmetic is round-to-nearest in a fixed order. */
int aps_ransac_sample_table(aps_ctx* ctx, const int64_t* pt_ptr, int64_t n_pairs, int64_t n_draws, uint64_t seed,
                            uint32_t* samples);
int aps_image_matching_batch(aps_ctx* ctx, int64_t n_pairs, const int64_t* pt_ptr, const double* pts1,
                             const double* pts2, double max_distance, double confidence, int max_trials,
                             const uint32_t* samples, int64_t n_draws, uint64_t seed, double* models,
                             double* models_inv, uint8_t* inliers, int32_t* n_inliers, uint8_t* accepted,
                             int32_t* draws_used);
/* Same, fed directly by the match lists (hand-off, SURVEY.md 8(f) rank 2): pair_ptr / rows = the CSR of the
 * n x n cell (aps_matchlist_pair_ptr / _rows), keypoints = pooled [F x 2] ROW-major doubles of all images,
 * img_off [n_images + 1], pairs_lin = find(candidatePairs) from aps_select_partners.  The matched points are
 * gathered on the device (refineMatch, imageMatching.m:224-227; out-of-range indices -> error id
 * refineMatch:MatchIndexOutOfBounds).  pt_ptr_out [n_pairs + 1] receives the offsets of each pair's
 * correspondences inside `inliers` (allMatches{ii,jj} = matches(inliers,:)). */
int aps_image_matching(aps_ctx* ctx, int n_images, const int64_t* pair_ptr, const uint32_t* rows,
                       const double* keypoints, const int64_t* img_off, const int64_t* pairs_lin, int64_t n_pairs,
                       double max_distance, double confidence, int max_trials, const uint32_t* samples,
                       int64_t n_draws, uint64_t seed, int64_t* pt_ptr_out, double* models, double* models_inv,
                       uint8_t* inliers, int32_t* n_inliers, uint8_t* accepted, int32_t* draws_used);
/* aps_image_matching for every candidate pair of nsets independent image sets in one pass.  pair_ptr[b] / rows[b] =
 * set b's CSR (what aps_matchlist_pair_ptr / _rows return for its list); keypoints = pooled [F x 2] ROW-major doubles of
 * all images of all sets (set 0's images first), img_off [sum n_b + 1]; set_pair_ptr / pairs_lin as
 * aps_select_partners_sets returns them.  Outputs are pooled in that pair order and mean what aps_image_matching's
 * mean: pt_ptr_out [n_pairs + 1] are offsets into the pooled `inliers`.  samples = [n_pairs x n_draws x 4] pooled in
 * the same order, or NULL to draw them on the device, pair p of set b keyed by p - set_pair_ptr[b] (its index in its
 * own set's list).  Every set's outputs are BIT-IDENTICAL to aps_image_matching on that set alone with the same seed.
 * Argument errors (checked before the context): nsets < 0, a negative image count or a bad pair index is APS_ERR_ARGS;
 * a match index outside a set's keypoints is refineMatch:MatchIndexOutOfBounds naming the set, and the call returns
 * nothing.  No limit on the number of pairs: the gather and the RANSAC chain run in chunks of at most 65535 pairs and
 * about 1 GiB of per-draw tables; launches grow with the chunks, never with nsets. */
int aps_image_matching_sets(aps_ctx* ctx, int nsets, const int* set_images, const int64_t* const* pair_ptr,
                            const uint32_t* const* rows, const double* keypoints, const int64_t* img_off,
                            const int64_t* set_pair_ptr, const int64_t* pairs_lin, double max_distance,
                            double confidence, int max_trials, const uint32_t* samples, int64_t n_draws,
                            uint64_t seed, int64_t* pt_ptr_out, double* models, double* models_inv,
                            uint8_t* inliers, int32_t* n_inliers, uint8_t* accepted, int32_t* draws_used);

/* ---- staged global pipeline (building block of the multi-GPU host; bench.py times these) -----
 * The stages of PP/featureMatching/featureMatchingGlobal.m as separate calls: pooling + normalisation :70-97
 * (create / upload), global kNN :106-120 (knn), per-feature filter loop :123-161 (filter, then compact after the
 * ranks exchanged their record slices).  All work is enqueued on the context's stream.  Query rows [q0,q1) of the pooled matrix may be
 * sharded across ranks: every rank holds all descriptors, so a query's neighbours are complete
 * locally and no cross-GPU merge exists (SURVEY.md 8(e)). */
int aps_gplan_create(aps_ctx* ctx, const int64_t* counts, int n, int D, int dtype, int k, aps_gplan** out);
void aps_gplan_destroy(aps_gplan* p);
int64_t aps_gplan_total(const aps_gplan* p); /* F */
/* Device pointer of the pooled ROW-major raw descriptor matrix [F x D] (float or uint8): fill it
 * with aps_gplan_upload(), or write it directly (device copy / ncclBroadcast) before prepare(). */
void* aps_gplan_desc_device(aps_gplan* p);
int aps_gplan_upload(aps_gplan* p, const void* const* desc, int layout); /* H2D + pooling (A1 :70-77) */
int aps_gplan_prepare(aps_gplan* p);                                     /* K1: A1 :80-97 */
int aps_gplan_knn(aps_gplan* p, int64_t q0, int64_t q1);                 /* K2/K3/K4: A2 */
int aps_gplan_filter(aps_gplan* p, int64_t q0, int64_t q1, double ratio); /* K5a: A3 :123-147 */
/* Per-query records written by filter(): [F + APS_RECORD_PAD] interleaved pairs (int32 target image, 1-based,
 * 0 = rejected ; uint32 partner = the match's local index in that image), 8 bytes per query row.  Rows outside
 * [q0,q1) are left untouched, so ranks exchange their slices with ONE in-place all-gather; the padding lets
 * equal-sized rank slices (multiples of 128 rows) run past F. */
#define APS_RECORD_PAD 16384
void* aps_gplan_records_device(aps_gplan* p);
/* Opt-in cross-check (NOT reference behaviour: featureMatchingGlobal.m:149-159 keeps A->B and B->A rows alike and
 * PP/mex/flann_knn.cpp:204 builds BFMatcher with crossCheck = false; BASELINE.json's "keeps mutual matches"): after
 * filter() on every rank's rows and the record exchange, a query keeps its match only if the matched feature's own
 * accepted match is that query.  Call between filter()/exchange and compact(). */
int aps_gplan_filter_mutual(aps_gplan* p);
void* aps_gplan_knn_idx_device(aps_gplan* p);  /* uint32 [F][k] row-major, 1-based */
void* aps_gplan_knn_dist_device(aps_gplan* p); /* float  [F][k] row-major */
/* D2H of the kNN table rows [q0,q1): idx/dist host buffers of (q1-q0)*k entries, row-major (synchronises) */
int aps_gplan_download_knn(aps_gplan* p, int64_t q0, int64_t q1, uint32_t* idx, float* dist);
int aps_gplan_compact(aps_gplan* p);                         /* K5b: A3 :149-159 on all F records */
int aps_gplan_download(aps_gplan* p, aps_matchlist** out);   /* D2H of the CSR lists (synchronises) */
int aps_gplan_pair_counts_device(aps_gplan* p, void** counts_i64); /* n*n int64, column-major, after compact() */

/* ---- staged pairwise pipeline (multi-GPU building block of featureMatchingPairwise; bench.py times these) ----
 * The reference broadcasts the descriptor cell to its parfor workers once and runs getMatches per pair
 * (PP/featureMatching/featureMatchingPairwise.m:48-59).  Here: descriptors uploaded (or written by a device producer /
 * an NCCL all-gather into aps_pplan_desc_device) once, K1 once (prepare), then match() computes this rank's share of
 * the column-major pair list -- pairs whose ordinal is congruent to pair_first modulo pair_stride -- with the
 * matchFeaturesScratch 'Exhaustive' semantics (:108-117, Unique = true). */
typedef struct aps_pplan aps_pplan;
int aps_pplan_create(aps_ctx* ctx, const int64_t* counts, int n, int D, int dtype, aps_pplan** out);
void aps_pplan_destroy(aps_pplan* p);
int64_t aps_pplan_total(const aps_pplan* p);
void* aps_pplan_desc_device(aps_pplan* p);   /* pooled ROW-major raw descriptors [F x D] */
int aps_pplan_upload(aps_pplan* p, const void* const* desc, int layout);
int aps_pplan_prepare(aps_pplan* p);
/* Matchingmethod / ApproxFloatNNMethod of getMatches (featureMatchingPairwise.m:108-117 -> matchFeaturesScratch.m:116-163).
 * Binary descriptors run the exhaustive Hamming search for every method, as the reference does (:611).  Float:
 *   APS_METHOD_EXHAUSTIVE            nearest2SSDExhaustive, D2 = a2 + b2' - 2 A B'                          (:322-366)
 *   APS_METHOD_APPROX_SUBSETPDIST2   pdist2(B(candB,:), A, 'euclidean', 'Smallest', 2), squared afterwards   (:149-155,
 *                                    :370-409); candB = ALL rows of B while N2 <= subset (12000, the reference's constant;
 *                                    PP/inputs.m:48 makes this the default).  Larger images: candB = `subset` distinct rows in
 *                                    a pseudo-random order drawn on the device from `seed` by a keyed bijection of [0, N2)
 *                                    -- a stand-in for randperm (MATLAB's stream cannot be reproduced), ONE subset per train
 *                                    image instead of one per call; aps_pplan_subset_table returns it (0-based rows of B)
 *   APS_METHOD_APPROX_KDTREE         knnsearch(createns(B,'kdtree'), A, 'K', 2): an EXACT Euclidean search, squared (:142-148)
 * Both approximate modes are served by the exact search with the Euclidean metric: distance = fl(sqrt(s))^2 with
 * s = sum((a-b).^2) in sequential float32, ranking by fl(sqrt(s)), ties -> lower index.
 *   APS_METHOD_APPROX_PCA2NN         nearest2ApproxFloatFast (:442-573): D > 48 -> PCA of the TRAIN image (mean, 48 leading
 *                                    components), both images projected, rows re-normalised, cosine similarity G = A*B',
 *                                    best = first maximum, second = maximum of the rest, d = 2 - 2 sim.  MathWorks' pca is
 *                                    closed source; restated with a fixed float64 covariance + cyclic Jacobi (csrc/aps_pca.cu)
 *                                    -- the similarities depend only on the 48-dimensional subspace, not on the basis. */
enum aps_method { APS_METHOD_EXHAUSTIVE = 0, APS_METHOD_APPROX_SUBSETPDIST2 = 1, APS_METHOD_APPROX_KDTREE = 2,
                  APS_METHOD_APPROX_PCA2NN = 3 };
int aps_pplan_set_method(aps_pplan* p, int method, int64_t subset, uint64_t seed);   /* before prepare() */
int aps_pplan_subset_table(aps_pplan* p, int image, int32_t* out /* [subset] */);   /* after prepare() */
int aps_pplan_match(aps_pplan* p, double match_threshold, double max_ratio, int pair_first, int pair_stride,
                    aps_matchlist** out);

/* ---- device group: single-process multi-GPU matching ------------------------------------------------------
 * The reference's only parallelism is parfor over the image pairs (PP/featureMatching/featureMatchingPairwise.m:48-59),
 * and a MATLAB process cannot join an NCCL world; a device group spreads one call of featureMatchingGlobal /
 * featureMatchingPairwise over several GPUs of one process instead.  The lists are BIT-IDENTICAL to the
 * single-context calls: the group runs the staged plans above on every member and exchanges only device buffers
 * (cudaMemcpyPeerAsync; staged by the driver where the GPUs have no peer access).  One host thread per member issues
 * that member's work, so the GPUs run concurrently even where the pairwise batches synchronise on host tables.
 * A one-member group runs exactly the single-context code on its device.
 *
 * aps_group_create: one aps_ctx per listed CUDA ordinal -- distinct and in range (else APS_ERR_ARGS), sm_100a (else
 *   APS_ERR_NOGPU, as without any device); where cudaDeviceCanAccessPeer allows, members get direct peer access to each
 *   other's memory, including their default stream-ordered memory pools (cudaMemPoolSetAccess), which hold every
 *   buffer the group exchanges.  This is process-wide state of those devices and is left in place by aps_group_destroy.
 * aps_group_ctx: member i's context (knobs such as aps_ctx_set_float_engine, and per-member statistics: after a global
 *   call aps_ctx_last_stats[0] of member i = the query rows it searched; after a pairwise call aps_ctx_pairwise_stats
 *   = its share of the screened pairs).
 * Failure of any member fails the whole call: no list is returned, every plan is released, and aps_last_error /
 * aps_error_id of the CALLING thread carry the first failing member's message and id. */
typedef struct aps_group aps_group;
int aps_group_create(const int* devices, int ndev, aps_group** out);
void aps_group_destroy(aps_group* g);
int aps_group_size(const aps_group* g);
aps_ctx* aps_group_ctx(aps_group* g, int i);
/* featureMatchingGlobal (float and uint8, k <= APS_MAX_K; mutual != 0 = the opt-in cross-check of
 * aps_gplan_filter_mutual).  Member i uploads a contiguous range of whole images (balanced by row count) and copies the
 * other members' ranges peer-to-peer, so every member holds all descriptors; K1 runs on every member; member i searches
 * query rows [q0, q1) = i-th block of equal multiples of 128 rows (members past F get an empty block) and filters them;
 * the record slices are copied into member 0, which cross-checks (if asked), compacts and downloads. */
int aps_group_feature_matching_global(aps_group* g, const void* const* desc, const int64_t* counts, int n, int D,
                                      int dtype, int layout, int k, double ratio, int mutual, aps_matchlist** out);
/* featureMatchingPairwise (float and uint8, every aps_method with its subset / seed as in aps_pplan_set_method).
 * Member 0 uploads; its pooled matrix is copied peer-to-peer to the other members; member i computes the pairs whose
 * column-major ordinal is congruent to i modulo the group size (aps_pplan_match(i, N)); the host lists are merged
 * into one CSR in cell order. */
int aps_group_feature_matching_pairwise(aps_group* g, const void* const* desc, const int64_t* counts, int n, int D,
                                        int dtype, int layout, double match_threshold, double max_ratio, int method,
                                        int64_t subset, uint64_t seed, aps_matchlist** out);
/* Measurement hook: member i's device time (ms, CUDA events on its stream) of the last multi-member call, per stage:
 * [0] host upload of its share, [1] peer exchange of the descriptors (includes waiting for the producers' uploads),
 * [2] search = K1 + kNN + filter (global) or K1 + its pair share (pairwise), [3] member 0 of a global call: from the
 * end of its own search to the lists on the host (waiting for the slowest member, record gather, cross-check,
 * compaction, download).  Stages a member did not run, and one-member groups, report 0. */
int aps_group_stage_times(aps_group* g, int i, double ms[4]);

/* ---- diagnostics (tests only): raw output of the tcgen05 candidate kernel -----------------------
 * Q [nq x D], T [nt x D] ROW-major float (used as given, no normalisation).  scores [nq x nt]
 * receives (bf16(q).bf16(t))*scale_t + bias_t as the kernel's epilogue computes it (scale = 1,
 * bias = -|t|^2/2); cand_idx / cand_score [nq x S x 8], S = aps_debug_tc_slots(ctx, nq, nt): the
 * candidate lists the kernel keeps per query row (one per column segment its work unit was split
 * into; 0-based train rows, 0xFFFFFFFF = empty).  Any of the three outputs may be NULL; nseg is ignored. */
int aps_debug_tc_slots(aps_ctx* ctx, int64_t nq, int64_t nt);
/* The fp16 screen of one pair: A [N1 x D], B [N2 x D] ROW-major float used as given.  b1b2 [N1 x 2] receives the two
 * values the screen keeps per query row (largest dot, and the second of the 8 column-class maxima); dump (may be NULL)
 * [N1 x dump_tiles x 64] the raw accumulator registers (two packed fp16 scores each) of the first dump_tiles tiles. */
int aps_debug_pair_screen(aps_ctx* ctx, const float* A, int64_t N1, const float* B, int64_t N2, int D, float* b1b2,
                          uint32_t* dump, int dump_tiles);
/* A device group of `nmembers` contexts that all live on `device` (aps_group_create refuses a repeated device): runs the
 * multi-member pipelines -- one host thread per member, event-ordered device-to-device exchanges, the merge -- on a
 * machine with one GPU.  The lists are the same as for any other group. */
int aps_debug_group_create_shared(int device, int nmembers, aps_group** out);
int aps_debug_tc_scores(aps_ctx* ctx, const float* Q, int64_t nq, const float* T, int64_t nt, int D, int nseg,
                        float* scores, uint32_t* cand_idx, float* cand_score);
/* The candidate lists of one tcgen05 launch, prepared and scheduled as the float searches run it.  Q [nq x D], T [nt x D]
 * ROW-major float; Q == T (and nq == nt) is a self-search.  prep 0: the global plan's preparation (rows normalised as
 * featureMatchingGlobal, fp16 operands, score = dot * scale); prep 1: flann_knn_win's (rows as given, bf16 operands,
 * score = dot - |t|^2/2).  The train view is sorted by scale unless natural_order.  Query rows [q0,q1) are searched
 * against train positions [t0,t1) of that view; rows != NULL runs the second pass of the search instead: the nrows
 * listed query rows (each inside [q0,q1)), gathered, every unit cut into column segments.
 * Outputs: cand_idx / cand_score with room for (q1-q0) x 32 entries, of which [(q1-q0) x nslot x 8] are written (row i
 * of the second pass = rows[i]): train-view positions (0xFFFFFFFF = empty) and packed scores, filled with 0xA5A5A5A5 /
 * NaN before the launch; perm [nt] train-view position -> row of T; q_bits [nq x D] and t_bits [nt x D]: the 16-bit
 * operands (fp16 or bf16) in the rows' original order; colscale / colbias [nt] per row of T.  info [11]: sm_count,
 * nslot, rows_full (leading rows whose candidates are all in list 0), operands-exact flag, operand kind (2 fp16, 0 bf16),
 * pre-filtered long sweep, units_full, tail_units, tail_seg, tail_balanced, tiles_per_seg. */
int aps_debug_tc_candidates(aps_ctx* ctx, const float* Q, int64_t nq, const float* T, int64_t nt, int D, int prep,
                            int natural_order, int64_t q0, int64_t q1, int64_t t0, int64_t t1, const int32_t* rows,
                            int64_t nrows, uint32_t* cand_idx, float* cand_score, int32_t* perm, uint16_t* q_bits,
                            uint16_t* t_bits, float* colscale, float* colbias, int64_t* info);
/* The same for the lists a search of k neighbours (1 <= k <= 12) keeps: K' = 8 candidates per list for k <= 5 (the
 * call above is this one with k = 4), 16 for 6 <= k <= 12.  cand_idx / cand_score need room for (q1-q0) x 64 entries,
 * of which [(q1-q0) x nslot x K'] are written.  info [12]: the 11 values above, then K'. */
int aps_debug_tc_candidates_k(aps_ctx* ctx, const float* Q, int64_t nq, const float* T, int64_t nt, int D, int prep,
                              int natural_order, int64_t q0, int64_t q1, int64_t t0, int64_t t1, const int32_t* rows,
                              int64_t nrows, uint32_t* cand_idx, float* cand_score, int32_t* perm, uint16_t* q_bits,
                              uint16_t* t_bits, float* colscale, float* colbias, int64_t* info, int k);

#ifdef __cplusplus
}
#endif
#endif /* APSMATCH_H */
