// aps_abi_internal.cuh -- what the translation units behind include/apsmatch.h share (aps_abi.cu: context, kNN entries,
// staged global pipeline; aps_abi_pairwise.cu: matchFeaturesScratch / featureMatchingPairwise, staged pairwise pipeline,
// pairwise matching of many image sets; aps_abi_sets.cu: global matching of many image sets).
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
int feature_matching_global_impl(aps_ctx* c, const void* const* desc, const int64_t* counts, int n, int D, int dtype,
                                 int layout, int k, double ratio, int mutual, aps_matchlist** out);
int feature_matching_pairwise_impl(aps_ctx* c, const void* const* desc, const int64_t* counts, int n, int D, int dtype,
                                   int layout, double match_threshold, double max_ratio, int method, int64_t subset,
                                   uint64_t seed, int pair_first, int pair_stride, aps_matchlist** out);

// ---- pooled upload of many images (aps_abi_sets.cu; the sets entries) ---------------------------------------------
// img[r] = image of pooled row r (d_off: [nimg + 1] row offsets on the device)
int sets_img_of_row(cudaStream_t s, const int64_t* d_off, int nimg, int64_t F, int32_t* img);
// H2D of image i (host ptrs[i], off[i + 1] - off[i] rows) to rows [off[i], off[i + 1]) of the pooled row-major matrix
// `raw`: one copy per image; column-major input is staged and transposed in ONE launch (needs img_of_row)
int sets_upload(aps_ctx* c, const void* const* ptrs, const std::vector<int64_t>& off, const int64_t* d_off,
                const int32_t* img_of_row, int D, int esz, int layout, void* raw);

// ---- match lists: the n x n cell in CSR form -----------------------------------------------------------------------
struct aps_matchlist {
  int n = 0;
  int64_t total = 0;
  std::vector<int64_t> pair_ptr;
  std::vector<uint32_t> rows;
  std::vector<double> metric;
  bool has_metric = false;
};
