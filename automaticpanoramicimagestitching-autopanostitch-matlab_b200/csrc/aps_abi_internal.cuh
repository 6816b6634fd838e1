// aps_abi_internal.cuh -- what the translation units behind include/apsmatch.h share (aps_abi.cu: context, kNN entries,
// staged global pipeline; aps_abi_pairwise.cu: matchFeaturesScratch / featureMatchingPairwise, staged pairwise pipeline,
// pairwise matching of many image sets; aps_abi_sets.cu: global matching of many image sets; aps_ransac.cu: RANSAC
// chunks; aps_global_image_matching.cu: global and pairwise matching through image matching in one call).
#pragma once
#include <string>
#include <vector>

#include "aps_common.cuh"

#define APS_FAIL(code, id, ...)            \
  do {                                     \
    aps_set_error(code, id, __VA_ARGS__);  \
    return code;                           \
  } while (0)

#define APS_CTX(c)                                                        \
  do {                                                                    \
    if (!(c)) APS_FAIL(APS_ERR_NOGPU, "apsmatch:nogpu", "context is NULL (no GPU context; there is no CPU path)"); \
    APS_CUDA(cudaSetDevice((c)->device));                                 \
  } while (0)

// ---- prepared float descriptor sets (aps_abi.cu) -----------------------------------------------------------------
struct FloatSide {          // one prepared descriptor set
  const float* raw = nullptr;  // [N x D]
  const float* xn = nullptr;   // normalised (or == raw)
  const float* sq = nullptr;   // sum(xn^2)
  const float* invn = nullptr;
  const __nv_bfloat16* xb = nullptr;  // [N x Dp] or nullptr when the tensor path is not prepared
  const float* colscale = nullptr;
  const float* colbias = nullptr;
  // train-side view of the tensor kernel (rows possibly sorted by scale, see aps_prep.cu)
  const __nv_bfloat16* xb_t = nullptr;
  const float* colscale_t = nullptr;
  const float* colbias_t = nullptr;
  const float4* tile_bounds = nullptr;
  const int32_t* perm = nullptr;  // sorted position -> original row (nullptr: identity)
  int64_t N = 0;
  int fp16 = 0;                   // operand rows are fp16 (flags[0] = exact in fp16) instead of bf16
};

// Prepared float set owning its buffers
struct FloatSet {
  DevBuf<float> raw, xn, sq, invn;
  DevBuf<__nv_bfloat16> xb;
  DevBuf<float> colscale, colbias;
  DevBuf<int32_t> flags;  // [8]: exact, maxdev bits, maxsq bits, maxabs bits
  // train-side view (floatset_finish_train)
  DevBuf<__nv_bfloat16> xb_t;
  DevBuf<float> colscale_t, colbias_t;
  DevBuf<int32_t> perm, sort_scratch;
  DevBuf<float4> tile_bounds;
  bool sorted = false;
  bool fp16 = false;  // tensor operands in fp16: 4x smaller rounding term than bf16; needs |x| inside the fp16 range
  int64_t N = 0;
  int D = 0;
  FloatSide side() const {
    FloatSide s;
    s.raw = raw.p;
    s.xn = xn.p ? xn.p : raw.p;
    s.sq = sq.p;
    s.invn = invn.p;
    s.xb = xb.p;
    s.colscale = colscale.p;
    s.colbias = colbias.p;
    s.xb_t = sorted ? xb_t.p : xb.p;
    s.colscale_t = sorted ? colscale_t.p : colscale.p;
    s.colbias_t = sorted ? colbias_t.p : colbias.p;
    s.tile_bounds = tile_bounds.p;
    s.perm = sorted ? perm.p : nullptr;
    s.N = N;
    s.fp16 = fp16 ? 1 : 0;
    return s;
  }
};

int floatset_alloc(aps_ctx* c, FloatSet& fs, int64_t N, int D);
int floatset_reset_flags(aps_ctx* c, FloatSet& fs);
int floatset_finish_train(aps_ctx* c, FloatSet& fs, bool sort);
int floatset_prepare(aps_ctx* c, FloatSet& fs, int norm_mode, bool tensor, int bias_mode, bool sort = true);
bool tc_wanted(const aps_ctx* c, int D, int64_t nq, int64_t nt, int k);
// metric 0: FLANN-order squared L2 (global path) ; metric 1: SSD (pairwise path)
int float_knn(aps_ctx* c, const FloatSide& Q, int64_t q0, int64_t q1, const FloatSide& T, int64_t t0, int64_t t1, int D,
              int k, int metric, int bias_mode, const int32_t* flags_dev, int64_t out_row0, uint32_t* idx, float* dist,
              bool use_tc);
int stage_matrix(aps_ctx* c, const void* host, int64_t N, int D, int esz, int layout, void* dst_rm, DevBuf<uint8_t>& tmp);
int pad_rows(cudaStream_t s, const uint8_t* src, int64_t N, int nb, int nb16, uint8_t* dst);
int hamming2_device(aps_ctx* c, const uint8_t* qpad, int64_t q0, int64_t N1, const uint8_t* tpad, int64_t t0, int64_t N2,
                    int nb, int nb16, uint32_t* idx2, float* d1, float* d2);
int ssd2_device(aps_ctx* c, const FloatSide& Q, int64_t q0, int64_t N1, const FloatSide& T, int64_t t0, int64_t N2, int D,
                const int32_t* flags, bool tc, int bias_mode, uint32_t* idx2, float* d1, float* d2);

// ---- one-call pipelines over the staged plans (aps_abi.cu / aps_abi_pairwise.cu; aps_abi_group.cu runs them per member)
int gplan_upload_images(aps_gplan* p, const void* const* desc, int layout, int i0, int i1);
// dev (here and below): desc[i] are device pointers into one pooled row-major matrix (pooled_image_ptrs), not host
// matrices in `layout`
int feature_matching_global_impl(aps_ctx* c, const void* const* desc, const int64_t* counts, int n, int D, int dtype,
                                 int layout, int k, double ratio, int mutual, aps_matchlist** out, bool dev = false);
int feature_matching_pairwise_impl(aps_ctx* c, const void* const* desc, const int64_t* counts, int n, int D, int dtype,
                                   int layout, double match_threshold, double max_ratio, int method, int64_t subset,
                                   uint64_t seed, int pair_first, int pair_stride, aps_matchlist** out,
                                   bool dev = false);

// ---- lists of image sets and pooled upload of many images (aps_abi_sets.cu; the sets entries) ---------------------
// Checks the set list of a sets entry (nsets >= 0, set_images[b] >= 0, at most INT_MAX images in all) and returns
// img0 [nsets + 1], the first pooled image of each set.  Messages number the sets from 1.
int sets_image_offsets(int nsets, const int* set_images, std::vector<int64_t>& img0);
// Splits a pooled match list whose cells are nsets column-major blocks (block j: cells [cell_off[j], cell_off[j + 1])
// of an n[j] x n[j] matrix) into one list per block, stored in out[slot[j]] (out[j] when slot is NULL).  metric: the
// pooled metric, or NULL for lists without one.
int sets_split_lists(int nsets, const std::vector<int64_t>& pair_ptr, const std::vector<uint32_t>& rows,
                     const std::vector<double>* metric, const std::vector<int64_t>& cell_off, const int* n,
                     const int* slot, aps_matchlist** out);
// img[r] = image of pooled row r (d_off: [nimg + 1] row offsets on the device)
int sets_img_of_row(cudaStream_t s, const int64_t* d_off, int nimg, int64_t F, int32_t* img);
// H2D of image i (host ptrs[i], off[i + 1] - off[i] rows) to rows [off[i], off[i + 1]) of the pooled row-major matrix
// `raw`: one copy per image; column-major input is staged and transposed in ONE launch (needs img_of_row).
// dev: ptrs[i] point into one pooled row-major device matrix; images whose rows follow each other there and in `raw`
// go in ONE device-to-device copy (one copy in all when the pass keeps the caller's image order)
int sets_upload(aps_ctx* c, const void* const* ptrs, const std::vector<int64_t>& off, const int64_t* d_off,
                const int32_t* img_of_row, int D, int esz, int layout, void* raw, bool dev = false);

// ---- device input (the *_dev entries) ------------------------------------------------------------------------------
// Per-image pointers into the pooled row-major device matrix d_pooled: image g starts at row sum(counts[0..g)).
std::vector<const void*> pooled_image_ptrs(const void* d_pooled, const int64_t* counts, int64_t nimg, int D, int esz);
// The checks and the hand-off of a *_dev entry once the host entry's statuses passed: d_pooled non-NULL when F > 0, the
// context, d_pooled (and d_kp when not NULL) device or managed memory; then the context's stream waits for an event
// recorded on producer_stream (when not NULL).
int dev_inputs(aps_ctx* c, int64_t F, const void* d_pooled, const void* d_kp, void* producer_stream);

// ---- global match lists kept on the device (aps_abi.cu, aps_abi_sets.cu; aps_global_image_matching_sets) ----------
// The compaction outputs of one global pass over nsets sets, in PASS order: pass position j is the caller's set
// order[j], its n x n block is cells [cell_off[j], cell_off[j + 1]) of pair_counts / pair_ptr (column-major, strict
// upper triangle filled), and cell c's rows are rows[2 * pair_ptr[c] .. 2 * pair_ptr[c + 1]).
struct GlobalLists {
  std::vector<int> order;
  std::vector<int64_t> cell_off;
  const int64_t* pair_counts = nullptr;  // [cells]
  const int64_t* pair_ptr = nullptr;     // [cells + 1]
  const uint32_t* rows = nullptr;
  const double* metric = nullptr;        // [rows] pairwise lists' metric (NULL: lists without one)
  DevBuf<int64_t> counts_buf, ptr_buf;   // owners for a pass over several sets
  DevBuf<uint32_t> rows_buf;
  DevBuf<double> metric_buf;
  aps_gplan* plan = nullptr;             // owner for one set
  int64_t F = 0, Ft = 0;                 // rows searched, rows of the tensor-path sets (statistics)
  GlobalLists() = default;
  GlobalLists(const GlobalLists&) = delete;
  GlobalLists& operator=(const GlobalLists&) = delete;
  ~GlobalLists() { aps_gplan_destroy(plan); }
};
// Checks the arguments of aps_feature_matching_global_sets (ids of aps_feature_matching_global) and returns the first
// pooled image of each set and the rows of each set.
int global_sets_args(int nsets, const int* set_images, const int64_t* counts, int D, int dtype, int k,
                     std::vector<int64_t>& img_first, std::vector<int64_t>& set_rows);
// Runs the global pass of aps_feature_matching_global_sets up to the compaction and leaves the lists on the device in
// L; the arguments must have passed global_sets_args, the context must be current and some set must have rows.
// Nothing is synchronised; global_lists_stats sets the context's statistics once the stream has been synchronised.
int global_lists_device(aps_ctx* c, int nsets, const int* set_images, const std::vector<int64_t>& img_first,
                        const std::vector<int64_t>& set_rows, const void* const* desc, const int64_t* counts, int D,
                        int dtype, int layout, int k, double ratio, int mutual, GlobalLists& L, bool dev = false);
void global_lists_stats(aps_ctx* c, int dtype, const GlobalLists& L);
// The one-set pass (aps_abi.cu): the staged plan from upload to compaction, and its lists handed to L.  dev: the
// plan's rows are one device-to-device copy from desc[0].
int gplan_run(aps_gplan* p, const void* const* desc, int layout, double ratio, int mutual, bool dev = false);
void gplan_lists(aps_gplan* p, GlobalLists& L);

// ---- pairwise match lists kept on the device (aps_abi_pairwise.cu; aps_pairwise_image_matching_sets) -------------
// The outputs of one pairwise pass over nsets sets, in the caller's set order: set j's n x n block is cells
// [cell_off[j], cell_off[j + 1]); rows / metric hold the M match rows in batch order.  The npairs pairs with rows are
// the table tab = [cell (npairs) | count (npairs) | src (npairs)]: pair q's rows are rows[2 * src[q] ..] and belong to
// cell cell[q].  Cells no pair names have no rows.
struct PairwiseRows {
  std::vector<int64_t> cell_off, tab;
  int64_t npairs = 0, M = 0;
  DevBuf<uint32_t> rows;
  DevBuf<double> metric;
};
// Checks the arguments of aps_feature_matching_pairwise_sets (its statuses) and returns the first pooled image of
// each set.
int pairwise_sets_args(int nsets, const int* set_images, const int64_t* counts, int D, int dtype, int method,
                       int64_t subset, std::vector<int64_t>& img_first);
// The pass of aps_feature_matching_pairwise_sets over every set (one set included) with its lists left on the device
// in R; the arguments must have passed pairwise_sets_args and the context must be current.  Its only synchronisations
// are those of the pass (the per-batch match counts among them); the pass's own buffers are released on return.
int pairwise_rows_device(aps_ctx* c, int nsets, const int* set_images, const void* const* desc, const int64_t* counts,
                         int nimg, int D, int dtype, int layout, double match_threshold, double max_ratio, int method,
                         int64_t subset, uint64_t seed, PairwiseRows& R, bool dev = false);

// ---- RANSAC over candidate pairs whose tables are on the device (aps_ransac.cu) ------------------------------------
// The gather and the RANSAC chain of aps_image_matching_sets over n_pairs pairs: pair p's correspondences are
// d_ptr[p] .. d_ptr[p + 1] of d_rows (packed 1-based match rows, images d_ii[p] / d_jj[p] of d_img_off / d_kp), its
// samples keyed by d_keys[p] (NULL: p).  Chunks of at most 65535 pairs and about 1 GiB of per-draw tables;
// ptr_host (may be NULL) lets chunks without correspondences skip the gather.  Outputs are device arrays.
int ransac_chunks(aps_ctx* c, int64_t n_pairs, int64_t total, const int64_t* d_ptr, const int64_t* ptr_host,
                  const uint32_t* d_rows, const int32_t* d_ii, const int32_t* d_jj, const int64_t* d_img_off,
                  const double2* d_kp, const int64_t* d_keys, const uint32_t* samples, int64_t n_draws, uint64_t seed,
                  double max_distance, double confidence, int max_trials, double* d_models, double* d_minv,
                  uint8_t* d_inl, int32_t* d_ni, uint8_t* d_acc, int32_t* d_used);
// pairs one chunk of ransac_chunks holds
int64_t ransac_chunk_pairs(int64_t n_draws);
int ransac_params(int64_t n_draws, int max_trials, double confidence);

// ---- match lists: the n x n cell in CSR form -----------------------------------------------------------------------
struct aps_matchlist {
  int n = 0;
  int64_t total = 0;
  std::vector<int64_t> pair_ptr;
  std::vector<uint32_t> rows;
  std::vector<double> metric;
  bool has_metric = false;
};
