// aps_abi_pairwise.cu -- the pairwise half of the extern "C" surface (include/apsmatch.h): matchFeaturesScratch for one
// pair, featureMatchingPairwise in one call, the staged pairwise pipeline aps_pplan_* (screen stage, exact stage,
// subset views of 'subsetpdist2', PCA views of 'pca2nn') and featureMatchingPairwise over many image sets in one call.
// No CPU compute path: without a CUDA device every entry fails.
#include <algorithm>
#include <chrono>
#include <climits>
#include <cstdlib>
#include <cmath>
#include <deque>
#include <limits>
#include <new>

#include "aps_abi_internal.cuh"

// ------------------------------------------------------------------------------------------------
// matchFeaturesScratch / featureMatchingPairwise
// One image pair of a pairwise pass; results are appended to the host vectors in the order of the pair list.
struct PairRef {
  int i, j;            // pooled image indices
  size_t ordinal;      // position in the pass's pair list
  int64_t qbase = -1;  // 'pca2nn': first row of the pair's projected query rows in the batch buffers (else: the image's rows)
  bool tensor = false; // the tensor engine (screen + tcgen05 candidates + exact re-rank) instead of the exact engine
};
// match lists of a pass, pair by pair: pair `ordinal` has cnt[ordinal] rows from row at[ordinal] of rows / metric (rows
// in batch order; one append per batch, no allocation per pair).  device: each batch's compacted rows and metric stay
// in their device buffers d_rows / d_met instead, and `at` counts rows over all batches (M so far).
struct PairResults {
  std::vector<int32_t> cnt;
  std::vector<int64_t> at;
  std::vector<uint32_t> rows;   // (col1, col2) per match
  std::vector<double> metric;
  bool device = false;
  int64_t M = 0;
  std::deque<DevBuf<uint32_t>> d_rows;
  std::deque<DevBuf<double>> d_met;
};
// 'pca2nn': the rows one pass of the pairwise pipeline reads when they are NOT the set's own -- the query rows of a batch
// projected with the train images' bases, and the projected train set
struct PcaViews {
  const float* q_xn; const float* q_sq; const float* q_invn; const void* q_xh; int64_t qN;
  const float* t_xn; const float* t_sq; const void* t_xh; int64_t tN;
  const float2* bounds;
  const int32_t* flags;
  int D;   // components kept (<= 48)
};

struct PairwiseSets {
  // per-image views: raw (un-normalised) and normalised (matchFeaturesScratch.m:105-110 is a
  // per-PAIR decision: normalise both iff max|A|>2 or max|B|>2)
  FloatSet rawset, normset;  // float
  DevBuf<uint8_t> u8raw, u8pad;
  int nb16 = 0;
  std::vector<int64_t> off;
  std::vector<int> big;  // per image: max|.| > 2
  // stage 1 (aps_pair_screen.cu): fp16 operand rows and per-image (min, max) squared norms of both views
  DevBuf<uint16_t> xh_raw, xh_norm;
  DevBuf<float> ones;    // [F + 256] column scales of the fp16 operand rows (they hold the values themselves: scale 1)
  DevBuf<float2> bounds_raw, bounds_norm;
  DevBuf<int64_t> d_img_off;
  // TRAIN VIEW.  Normally the set's own rows.  'subsetpdist2' with images above the subset size: extended copies whose
  // rows [Freal, Freal + nbig * vcnt) hold, per big image, the rows candB = randperm-like subset (a "virtual image").
  int64_t Freal = 0, vcnt = 0;
  std::vector<int64_t> voff;   // per image: first row of its virtual image in the train view, -1 = use the real rows
  DevBuf<int32_t> vsrc, vmap, d_big;
  DevBuf<float> tv_xn[2], tv_sq[2], tv_colbias[2], tv_ones;   // [0] un-normalised view, [1] normalised view
  DevBuf<uint16_t> tv_xh[2];
  DevBuf<int64_t> d_tstart, d_tcount;
  // 'pca2nn' (aps_pca.cu): per view [0] un-normalised / [1] normalised: basis of every image and the projected,
  // normalised train rows [F x P] with their fp16 operands [F x 64]
  int pcaP = 0;
  DevBuf<float> pca_mu[2], pca_coeff[2], pca_txn[2], pca_tsq[2], pca_tinvn[2];
  DevBuf<uint16_t> pca_txh[2];
  DevBuf<float2> pca_bounds[2];
  DevBuf<int32_t> pca_flags[2];
  bool subsets() const { return !voff.empty(); }
  int64_t toff(int j) const { return (subsets() && voff[j] >= 0) ? voff[j] : off[j]; }
  int64_t tcnt(int j, const int64_t* counts) const { return (subsets() && voff[j] >= 0) ? vcnt : counts[j]; }
};

// what the pairwise kernels read on the train side
struct TrainView {
  const float* xn;
  const float* sq;
  const void* xh;
  const float* colbias;
  const float* ones;
  int64_t N;
};
static TrainView train_view(const PairwiseSets& ps, bool norm) {
  const FloatSet& S = norm ? ps.normset : ps.rawset;
  TrainView v;
  const int w = norm ? 1 : 0;
  if (ps.subsets() && ps.tv_xn[w].p) {
    v.xn = ps.tv_xn[w].p; v.sq = ps.tv_sq[w].p; v.xh = ps.tv_xh[w].p; v.colbias = ps.tv_colbias[w].p; v.ones = ps.tv_ones.p;
    v.N = ps.Freal + (int64_t)ps.vcnt * (int64_t)(ps.vsrc.n / (ps.vcnt > 0 ? ps.vcnt : 1));
  } else {
    v.xn = S.xn.p ? S.xn.p : S.raw.p; v.sq = S.sq.p; v.xh = norm ? (const void*)ps.xh_norm.p : (const void*)ps.xh_raw.p;
    v.colbias = S.colbias.p; v.ones = ps.ones.p; v.N = S.N;
  }
  return v;
}

// allocation of the pooled raw matrix + bookkeeping
static int pairwise_alloc(aps_ctx* c, PairwiseSets& ps, const int64_t* counts, int n, int D, int dtype) {
  ps.off.assign(n + 1, 0);
  ps.big.assign(n, 0);
  for (int i = 0; i < n; ++i) ps.off[i + 1] = ps.off[i] + counts[i];
  const int64_t F = ps.off[n];
  if (dtype == APS_F32) {
    APS_TRY(floatset_alloc(c, ps.rawset, F, D));
  } else {
    ps.nb16 = (D + 15) / 16 * 16;
    APS_TRY(ps.u8raw.alloc((size_t)F * D, c->stream));
    APS_TRY(ps.u8pad.alloc((size_t)F * ps.nb16, c->stream));
  }
  return APS_OK;
}

// H2D of the per-image matrices into the pooled row-major matrix (vertcat of the cell)
static int pairwise_upload(aps_ctx* c, PairwiseSets& ps, const void* const* desc, const int64_t* counts, int n, int D,
                           int dtype, int layout) {
  const int64_t F = ps.off[n];
  const int esz = dtype == APS_F32 ? 4 : 1;
  char* base = dtype == APS_F32 ? (char*)ps.rawset.raw.p : (char*)ps.u8raw.p;
  DevBuf<uint8_t> stage;
  if (layout == APS_COL_MAJOR && F > 0) APS_TRY(stage.alloc((size_t)F * D * esz, c->stream));
  for (int i = 0; i < n; ++i) {
    if (counts[i] == 0) continue;
    if (!desc || !desc[i]) APS_FAIL(APS_ERR_ARGS, "", "descriptor pointer %d is NULL", i);
    char* dst = base + (size_t)ps.off[i] * D * esz;
    size_t bytes = (size_t)counts[i] * D * esz;
    if (layout == APS_ROW_MAJOR) {
      APS_CUDA(cudaMemcpyAsync(dst, desc[i], bytes, cudaMemcpyHostToDevice, c->stream));
    } else {
      char* st = (char*)stage.p + (size_t)ps.off[i] * D * esz;
      APS_CUDA(cudaMemcpyAsync(st, desc[i], bytes, cudaMemcpyHostToDevice, c->stream));
      APS_TRY(aps_k_transpose_in(c->stream, st, counts[i], D, esz, dst));
    }
  }
  return APS_OK;
}

// K1 of the pairwise path: per-image magnitude test (normalise iff max|.| > 2 is a per-PAIR decision,
// matchFeaturesScratch.m:105-110), row norms, tensor operands of the raw and (when needed) the normalised view
static int pairwise_finish(aps_ctx* c, PairwiseSets& ps, const int64_t* counts, int n, int D, int dtype, bool tensor) {
  const int64_t F = ps.off[n];
  if (dtype == APS_U8) {
    APS_TRY(pad_rows(c->stream, ps.u8raw.p, F, D, ps.nb16, ps.u8pad.p));
    return APS_OK;
  }
  if (F == 0) return APS_OK;
  // per-image max|.|: run the norm pass image by image with its own flag words
  DevBuf<int32_t> imgflags;
  APS_TRY(imgflags.alloc((size_t)n * 8, c->stream));
  std::vector<int32_t> init((size_t)n * 8, 0);
  for (int i = 0; i < n; ++i) init[(size_t)i * 8] = 1;
  APS_CUDA(cudaMemcpyAsync(imgflags.p, init.data(), init.size() * 4, cudaMemcpyHostToDevice, c->stream));
  int64_t maxc = 0;
  for (int i = 0; i < n; ++i) maxc = counts[i] > maxc ? counts[i] : maxc;
  APS_TRY(ps.d_img_off.alloc((size_t)n + 1, c->stream));
  APS_CUDA(cudaMemcpyAsync(ps.d_img_off.p, ps.off.data(), (size_t)(n + 1) * 8, cudaMemcpyHostToDevice, c->stream));
  APS_TRY(aps_k_prepare_norm_images(c->stream, ps.rawset.raw.p, ps.d_img_off.p, n, maxc, D, APS_NORM_NONE, ps.rawset.raw.p,
                                    ps.rawset.sq.p, ps.rawset.invn.p, imgflags.p));
  std::vector<int32_t> hf((size_t)n * 8);
  APS_CUDA(cudaMemcpyAsync(hf.data(), imgflags.p, hf.size() * 4, cudaMemcpyDeviceToHost, c->stream));
  APS_CUDA(cudaStreamSynchronize(c->stream));
  ps.big.assign(n, 0);
  bool any_big = false, all_exact = true;
  for (int i = 0; i < n; ++i) {
    if (counts[i] == 0) continue;
    float maxabs;
    memcpy(&maxabs, &hf[(size_t)i * 8 + 3], 4);
    ps.big[i] = maxabs > 2.0f;
    any_big |= ps.big[i] != 0;
    all_exact &= hf[(size_t)i * 8] != 0;
  }
  // flag words shared by all images of a view (exactness must hold on both sides of every pair)
  {
    int32_t fl[8] = {all_exact ? 1 : 0, 0, 0, 0, 0, 0, 0, 0};
    for (int i = 0; i < n; ++i)   // max over the images of the magnitude words (bit patterns of non-negative floats)
      for (int w = 1; w < 4; ++w)
        if (counts[i] > 0 && hf[(size_t)i * 8 + w] > fl[w]) fl[w] = hf[(size_t)i * 8 + w];
    APS_CUDA(cudaMemcpyAsync(ps.rawset.flags.p, fl, sizeof fl, cudaMemcpyHostToDevice, c->stream));
    APS_CUDA(cudaStreamSynchronize(c->stream));
  }
  if (tensor) {
    const int Dp = (D + 63) / 64 * 64;
    APS_TRY(ps.rawset.xb.alloc((size_t)F * Dp, c->stream));
    APS_TRY(ps.rawset.colscale.alloc((size_t)F + 256, c->stream));
    APS_TRY(ps.rawset.colbias.alloc((size_t)F + 256, c->stream));
    APS_TRY(aps_k_prepare_operands(c->stream, ps.rawset.raw.p, ps.rawset.raw.p, ps.rawset.sq.p, ps.rawset.invn.p, F,
                                   D, Dp, ps.rawset.flags.p, 1, ps.rawset.xb.p, ps.rawset.colscale.p, ps.rawset.colbias.p));
    APS_TRY(floatset_finish_train(c, ps.rawset, /*sort*/ false));  // image ranges must stay contiguous
    APS_TRY(ps.xh_raw.alloc((size_t)F * Dp, c->stream));
    APS_TRY(ps.bounds_raw.alloc((size_t)n, c->stream));
    APS_TRY(ps.ones.alloc((size_t)F + 256, c->stream));
    APS_TRY(aps_k_fill_f32(c->stream, ps.ones.p, F + 256, 1.0f));
    APS_TRY(aps_k_prepare_operands_f16(c->stream, ps.rawset.raw.p, F, D, Dp, ps.xh_raw.p));
  }
  if (any_big) {
    APS_TRY(floatset_alloc(c, ps.normset, F, D));
    APS_TRY(floatset_reset_flags(c, ps.normset));
    APS_CUDA(cudaMemcpyAsync(ps.normset.raw.p, ps.rawset.raw.p, (size_t)F * D * 4, cudaMemcpyDeviceToDevice, c->stream));
    // normalised rows: scale-only scoring (bias would have to be scaled per query row)
    APS_TRY(floatset_prepare(c, ps.normset, APS_NORM_PAIRWISE, tensor, 0, /*sort*/ false));
    if (tensor) {
      const int Dp = (D + 63) / 64 * 64;
      APS_TRY(ps.xh_norm.alloc((size_t)F * Dp, c->stream));
      APS_TRY(ps.bounds_norm.alloc((size_t)n, c->stream));
      APS_TRY(aps_k_prepare_operands_f16(c->stream, ps.normset.xn.p, F, D, Dp, ps.xh_norm.p));
    }
  }
  return APS_OK;
}

// Train view of the staged plan (after pairwise_finish): per-image norm bounds of the screen, and -- for 'subsetpdist2'
// with images above `subset` rows -- the virtual subset images (matchFeaturesScratch.m:388-393: candB = randperm(N2,
// subset), B2 = B(candB,:); here ONE subset per train image, drawn by a keyed bijection, instead of one per call).
// key[j] (nullptr: j) keys image j's subset: its index in its own set.
static int pairwise_build_train_view(aps_ctx* c, PairwiseSets& ps, const int64_t* counts, int n, int D, bool tensor,
                                     int64_t subset, uint64_t seed, const int32_t* key = nullptr) {
  cudaStream_t s = c->stream;
  const int64_t F = ps.off[n];
  ps.Freal = F;
  ps.voff.clear();
  ps.vcnt = 0;
  if (F == 0) return APS_OK;
  std::vector<int32_t> big;
  if (subset > 0)
    for (int j = 0; j < n; ++j)
      if (counts[j] > subset) big.push_back(j);
  const int Dp = (D + 63) / 64 * 64;
  if (!big.empty()) {
    const int nbig = (int)big.size();
    const int64_t V = (int64_t)nbig * subset;
    if (F + V >= ((int64_t)1 << 31) - 512) APS_FAIL(APS_ERR_ARGS, "", "too many descriptors for the subset views");
    ps.voff.assign(n, -1);
    ps.vcnt = subset;
    for (int b = 0; b < nbig; ++b) ps.voff[big[b]] = F + (int64_t)b * subset;
    for (int b = 0; b < nbig; ++b) big.push_back(key ? key[big[b]] : big[b]);   // [nbig, 2 nbig): key indices
    APS_TRY(ps.d_big.alloc((size_t)nbig * 2, s));
    APS_TRY(ps.vsrc.alloc((size_t)V, s));
    APS_TRY(ps.vmap.alloc((size_t)V, s));
    APS_CUDA(cudaMemcpyAsync(ps.d_big.p, big.data(), (size_t)nbig * 8, cudaMemcpyHostToDevice, s));
    APS_CUDA(cudaStreamSynchronize(s));   // `big` is pageable host memory
    APS_TRY(aps_k_subset_rows(s, ps.d_img_off.p, ps.d_big.p, ps.d_big.p + nbig, nbig, subset, seed, ps.vsrc.p,
                              ps.vmap.p));
    APS_TRY(ps.tv_ones.alloc((size_t)(F + V) + 256, s));
    APS_TRY(aps_k_fill_f32(s, ps.tv_ones.p, F + V + 256, 1.0f));
    for (int w = 0; w < 2; ++w) {
      const FloatSet& S = w ? ps.normset : ps.rawset;
      if (S.N == 0) continue;
      const float* xn = S.xn.p ? S.xn.p : S.raw.p;
      const uint16_t* xh = w ? ps.xh_norm.p : ps.xh_raw.p;
      APS_TRY(ps.tv_xn[w].alloc((size_t)(F + V) * D, s));
      APS_TRY(ps.tv_sq[w].alloc((size_t)(F + V), s));
      APS_CUDA(cudaMemcpyAsync(ps.tv_xn[w].p, xn, (size_t)F * D * 4, cudaMemcpyDeviceToDevice, s));
      APS_CUDA(cudaMemcpyAsync(ps.tv_sq[w].p, S.sq.p, (size_t)F * 4, cudaMemcpyDeviceToDevice, s));
      APS_TRY(aps_k_gather_f32_rows(s, xn, ps.vsrc.p, V, D, ps.tv_xn[w].p + (size_t)F * D));
      APS_TRY(aps_k_gather_f32_rows(s, S.sq.p, ps.vsrc.p, V, 1, ps.tv_sq[w].p + F));
      if (tensor && xh) {
        APS_TRY(ps.tv_xh[w].alloc((size_t)(F + V) * Dp, s));
        APS_TRY(ps.tv_colbias[w].alloc((size_t)(F + V) + 256, s));
        APS_CUDA(cudaMemcpyAsync(ps.tv_xh[w].p, xh, (size_t)F * Dp * 2, cudaMemcpyDeviceToDevice, s));
        APS_TRY(aps_k_gather_u16_rows(s, xh, ps.vsrc.p, V, Dp, ps.tv_xh[w].p + (size_t)F * Dp));
        APS_CUDA(cudaMemsetAsync(ps.tv_colbias[w].p, 0, ((size_t)(F + V) + 256) * 4, s));
        if (S.colbias.p) {
          APS_CUDA(cudaMemcpyAsync(ps.tv_colbias[w].p, S.colbias.p, (size_t)F * 4, cudaMemcpyDeviceToDevice, s));
          APS_TRY(aps_k_gather_f32_rows(s, S.colbias.p, ps.vsrc.p, V, 1, ps.tv_colbias[w].p + F));
        }
      }
    }
  }
  if (tensor) {   // per TRAIN image (real rows or its subset): (min, max) of the squared norms, for the screen's bounds
    std::vector<int64_t> st((size_t)n * 2);
    for (int j = 0; j < n; ++j) {
      st[j] = ps.toff(j);
      st[(size_t)n + j] = ps.tcnt(j, counts);
    }
    APS_TRY(ps.d_tstart.alloc((size_t)n * 2, s));
    APS_CUDA(cudaMemcpyAsync(ps.d_tstart.p, st.data(), st.size() * 8, cudaMemcpyHostToDevice, s));
    APS_CUDA(cudaStreamSynchronize(s));
    for (int w = 0; w < 2; ++w) {
      const FloatSet& S = w ? ps.normset : ps.rawset;
      DevBuf<float2>& bo = w ? ps.bounds_norm : ps.bounds_raw;
      if (S.N == 0 || !bo.p) continue;
      const TrainView tv = train_view(ps, w == 1);
      APS_TRY(aps_k_image_sq_bounds(s, tv.sq, ps.d_tstart.p, ps.d_tstart.p + n, n, bo.p));
    }
  }
  return APS_OK;
}

// 'pca2nn' (matchFeaturesScratch.m:130-141, 442-573): per view, the PCA basis of every image (it is the TRAIN image's basis
// that a pair uses, :476-483), the projected + re-normalised (:486-487) train rows and their fp16 operands.  D <= 48: no
// PCA (:477), the rows are only re-normalised -- expressed as the identity basis so that one code path serves both.
__global__ void k_identity_basis(int n, int D, float* __restrict__ mu, float* __restrict__ coeff) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < (int64_t)n * D) mu[i] = 0.f;
  if (i < (int64_t)n * D * D) {
    const int64_t e = i % ((int64_t)D * D);
    coeff[i] = (e / D == e % D) ? 1.f : 0.f;
  }
}
static int pairwise_build_pca(aps_ctx* c, PairwiseSets& ps, const int64_t* counts, int n, int D) {
  cudaStream_t s = c->stream;
  const int64_t F = ps.off[n];
  if (F == 0) return APS_OK;
  const int P = D > aps_pca_components() ? aps_pca_components() : D;
  ps.pcaP = P;
  for (int w = 0; w < 2; ++w) {
    const FloatSet& S = w ? ps.normset : ps.rawset;
    if (S.N == 0 || !S.raw.p) continue;
    const float* X = S.xn.p ? S.xn.p : S.raw.p;
    APS_TRY(ps.pca_mu[w].alloc((size_t)n * D, s));
    APS_TRY(ps.pca_coeff[w].alloc((size_t)n * D * P, s));
    if (D > aps_pca_components()) {
      DevBuf<double> scratch;
      APS_TRY(scratch.alloc((size_t)2 * n * D * D, s));
      APS_TRY(aps_k_pca_basis(s, X, ps.d_img_off.p, n, D, P, ps.pca_mu[w].p, ps.pca_coeff[w].p, scratch.p));
    } else {
      k_identity_basis<<<(unsigned)aps_ceil_div((int64_t)n * D * D, 256), 256, 0, s>>>(n, D, ps.pca_mu[w].p, ps.pca_coeff[w].p);
      APS_LAUNCHED();
    }
    std::vector<aps_proj_seg> segs;
    for (int j = 0; j < n; ++j)
      if (counts[j] > 0) segs.push_back(aps_proj_seg{ps.off[j], ps.off[j], (int32_t)counts[j], j});
    APS_TRY(ps.pca_txn[w].alloc((size_t)F * P, s));
    APS_TRY(ps.pca_tsq[w].alloc((size_t)F, s));
    APS_TRY(ps.pca_tinvn[w].alloc((size_t)F, s));
    APS_TRY(ps.pca_txh[w].alloc((size_t)F * 64, s));
    APS_TRY(ps.pca_bounds[w].alloc((size_t)n, s));
    APS_TRY(ps.pca_flags[w].alloc(8, s));
    static const int32_t init[8] = {1, 0, 0, 0, 0, 0, 0, 0};
    APS_CUDA(cudaMemcpyAsync(ps.pca_flags[w].p, init, sizeof init, cudaMemcpyHostToDevice, s));
    APS_TRY(aps_k_pca_project(s, X, D, P, segs, ps.pca_mu[w].p, ps.pca_coeff[w].p, ps.pca_txn[w].p));
    APS_TRY(aps_k_prepare_norm(s, ps.pca_txn[w].p, F, P, APS_NORM_PAIRWISE, ps.pca_txn[w].p, ps.pca_tsq[w].p,
                               ps.pca_tinvn[w].p, ps.pca_flags[w].p, 1));
    APS_TRY(aps_k_prepare_operands_f16(s, ps.pca_txn[w].p, F, P, 64, ps.pca_txh[w].p));
    std::vector<int64_t> st((size_t)n * 2);
    for (int j = 0; j < n; ++j) {
      st[j] = ps.off[j];
      st[(size_t)n + j] = counts[j];
    }
    DevBuf<int64_t> d_st;
    APS_TRY(d_st.alloc(st.size(), s));
    APS_CUDA(cudaMemcpyAsync(d_st.p, st.data(), st.size() * 8, cudaMemcpyHostToDevice, s));
    APS_CUDA(cudaStreamSynchronize(s));
    APS_TRY(aps_k_image_sq_bounds(s, ps.pca_tsq[w].p, d_st.p, d_st.p + n, n, ps.pca_bounds[w].p));
  }
  return APS_OK;
}

// one batch of pairs in 'pca2nn' mode: project the query rows with their train images' bases, re-normalise, screen, match
static int pairwise_screen_stage(aps_ctx* c, PairwiseSets& ps, std::vector<PairRef>& pairs, const int64_t* counts, int D,
                                 bool norm, double match_threshold, double max_ratio, const PcaViews* pv = nullptr);
static int pairwise_batch(aps_ctx* c, PairwiseSets& ps, const std::vector<PairRef>& pairs, const int64_t* counts, int D,
                          int dtype, bool norm, bool tensor, int dist_metric, double match_threshold, double max_ratio,
                          PairResults& res, const PcaViews* pv = nullptr);
static int pairwise_pca_batch(aps_ctx* c, PairwiseSets& ps, std::vector<PairRef> batch, const int64_t* counts, int D,
                              bool norm, bool tensor, double match_threshold, double max_ratio, PairResults& res) {
  cudaStream_t s = c->stream;
  const int w = norm ? 1 : 0, P = ps.pcaP;
  const FloatSet& S = norm ? ps.normset : ps.rawset;
  const float* X = S.xn.p ? S.xn.p : S.raw.p;
  std::vector<aps_proj_seg> segs;
  int64_t E = 0;
  for (PairRef& pr : batch) {
    pr.qbase = E;
    segs.push_back(aps_proj_seg{ps.off[pr.i], E, (int32_t)counts[pr.i], pr.j});
    E += counts[pr.i];
  }
  if (E == 0) return APS_OK;
  DevBuf<float> qxn, qsq, qinvn;
  DevBuf<uint16_t> qxh;
  APS_TRY(qxn.alloc((size_t)E * P, s));
  APS_TRY(qsq.alloc((size_t)E, s));
  APS_TRY(qinvn.alloc((size_t)E, s));
  APS_TRY(aps_k_pca_project(s, X, D, P, segs, ps.pca_mu[w].p, ps.pca_coeff[w].p, qxn.p));
  APS_TRY(aps_k_prepare_norm(s, qxn.p, E, P, APS_NORM_PAIRWISE, qxn.p, qsq.p, qinvn.p, ps.pca_flags[w].p, 1));
  PcaViews pv;
  pv.q_xn = qxn.p; pv.q_sq = qsq.p; pv.q_invn = qinvn.p; pv.q_xh = nullptr; pv.qN = E;
  pv.t_xn = ps.pca_txn[w].p; pv.t_sq = ps.pca_tsq[w].p; pv.t_xh = ps.pca_txh[w].p; pv.tN = ps.off.back();
  pv.bounds = ps.pca_bounds[w].p; pv.flags = ps.pca_flags[w].p; pv.D = P;
  if (tensor) {
    APS_TRY(qxh.alloc((size_t)E * 64, s));
    APS_TRY(aps_k_prepare_operands_f16(s, qxn.p, E, P, 64, qxh.p));
    pv.q_xh = qxh.p;
    if (c->pairwise_screen) APS_TRY(pairwise_screen_stage(c, ps, batch, counts, D, norm, match_threshold, max_ratio, &pv));
  }
  return pairwise_batch(c, ps, batch, counts, D, APS_F32, norm, tensor, /*metric*/ 3, match_threshold, max_ratio, res, &pv);
}

static int pairwise_prepare(aps_ctx* c, PairwiseSets& ps, const void* const* desc, const int64_t* counts, int n,
                            int D, int dtype, int layout, bool tensor) {
  APS_TRY(pairwise_alloc(c, ps, counts, n, D, dtype));
  APS_TRY(pairwise_upload(c, ps, desc, counts, n, D, dtype, layout));
  APS_TRY(pairwise_finish(c, ps, counts, n, D, dtype, tensor));
  if (dtype == APS_F32) APS_TRY(pairwise_build_train_view(c, ps, counts, n, D, tensor, 0, 0));
  return APS_OK;
}

// one pair on the device: results into caller regions; count stays on the device
static int pair_device(aps_ctx* c, PairwiseSets& ps, int i, int j, const int64_t* counts, int D, int dtype,
                       double match_threshold, double max_ratio, int unique, bool tensor, uint32_t* matches,
                       double* metric, int32_t* count_dev) {
  const int64_t N1 = counts[i], N2 = counts[j];
  if (N1 == 0 || N2 == 0) {  // matchFeaturesScratch.m:84-88 (binary); float: documented deviation
    APS_CUDA(cudaMemsetAsync(count_dev, 0, sizeof(int32_t), c->stream));
    return APS_OK;
  }
  DevBuf<uint32_t> idx2;
  DevBuf<float> d1, d2;
  DevBuf<unsigned long long> best, keys;
  APS_TRY(idx2.alloc((size_t)N1, c->stream));
  APS_TRY(d1.alloc((size_t)N1, c->stream));
  APS_TRY(d2.alloc((size_t)N1, c->stream));
  APS_TRY(best.alloc((size_t)N2, c->stream));
  APS_TRY(keys.alloc((size_t)N1 * 2, c->stream));
  if (dtype == APS_U8) {
    APS_TRY(hamming2_device(c, ps.u8pad.p, ps.off[i], N1, ps.u8pad.p, ps.off[j], N2, D, ps.nb16, idx2.p, d1.p, d2.p));
    APS_TRY(aps_k_pair_filter_unique(c->stream, idx2.p, d1.p, d2.p, N1, N2, 1, D * 8, match_threshold, max_ratio,
                                     unique, best.p, keys.p, count_dev, matches, metric));
  } else {
    const bool norm = ps.big[i] || ps.big[j];
    FloatSet& S = norm ? ps.normset : ps.rawset;
    FloatSide side = S.side();
    APS_TRY(ssd2_device(c, side, ps.off[i], N1, side, ps.off[j], N2, D, S.flags.p, tensor, norm ? 0 : 1, idx2.p,
                        d1.p, d2.p));
    APS_TRY(aps_k_pair_filter_unique(c->stream, idx2.p, d1.p, d2.p, N1, N2, 0, 0, match_threshold, max_ratio,
                                     unique, best.p, keys.p, count_dev, matches, metric));
  }
  return APS_OK;
}

extern "C" int aps_match_features(aps_ctx* c, const void* F1, int64_t N1, const void* F2, int64_t N2, int D,
                                  int dtype, int layout, double match_threshold, double max_ratio, int unique,
                                  uint32_t* matches, double* metric, int64_t* K) {
  APS_CTX(c);
  if (!K) APS_FAIL(APS_ERR_ARGS, "", "K is NULL");
  *K = 0;
  if (dtype != APS_F32 && dtype != APS_U8) APS_FAIL(APS_ERR_TYPE, "", "descriptors must be single or uint8");
  if (N1 == 0 || N2 == 0) return APS_OK;
  if (!F1 || !F2 || !matches || !metric) APS_FAIL(APS_ERR_ARGS, "", "null pointer argument");
  if (D <= 0) APS_FAIL(APS_ERR_DIM, "", "descriptor dimension must be positive");
  c->stats[0] = c->stats[1] = c->stats[2] = c->stats[3] = 0;
  const void* desc[2] = {F1, F2};
  const int64_t counts[2] = {N1, N2};
  const bool tensor = dtype == APS_F32 && tc_wanted(c, D, N1, N2, 2);
  PairwiseSets ps;
  APS_TRY(pairwise_prepare(c, ps, desc, counts, 2, D, dtype, layout, tensor));
  DevBuf<uint32_t> dm;
  DevBuf<double> dmet;
  DevBuf<int32_t> cnt;
  APS_TRY(dm.alloc((size_t)N1 * 2, c->stream));
  APS_TRY(dmet.alloc((size_t)N1, c->stream));
  APS_TRY(cnt.alloc(1, c->stream));
  APS_TRY(pair_device(c, ps, 0, 1, counts, D, dtype, match_threshold, max_ratio, unique, tensor, dm.p, dmet.p, cnt.p));
  int32_t hk = 0;
  APS_CUDA(cudaMemcpyAsync(&hk, cnt.p, 4, cudaMemcpyDeviceToHost, c->stream));
  APS_CUDA(cudaStreamSynchronize(c->stream));
  if (hk > 0) {
    APS_CUDA(cudaMemcpyAsync(matches, dm.p, (size_t)hk * 8, cudaMemcpyDeviceToHost, c->stream));
    APS_CUDA(cudaMemcpyAsync(metric, dmet.p, (size_t)hk * 8, cudaMemcpyDeviceToHost, c->stream));
    APS_CUDA(cudaStreamSynchronize(c->stream));
  }
  *K = hk;
  c->stats[1] = c->h_flags[32];
  return APS_OK;
}


// packBits (matchFeaturesScratch.m:617-646): [N x Dbits] 0/1 bytes -> [N x ceil(Dbits/8)] bytes, MSB first
__global__ void k_pack_bits01(const uint8_t* __restrict__ bits, int64_t N, int Dbits, int nb, uint8_t* __restrict__ packed) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N * nb) return;
  const int64_t r = i / nb;
  const int byte = (int)(i - r * nb);
  unsigned v = 0;
  for (int b = 0; b < 8; ++b) {
    const int col = byte * 8 + b;
    if (col < Dbits && bits[r * Dbits + col]) v |= 1u << (7 - b);
  }
  packed[i] = (uint8_t)v;
}

extern "C" int aps_match_features_bits(aps_ctx* c, const uint8_t* F1, int64_t N1, const uint8_t* F2, int64_t N2,
                                       int Dbits, int layout, double match_threshold, double max_ratio, int unique,
                                       uint32_t* matches, double* metric, int64_t* K) {
  APS_CTX(c);
  if (!K) APS_FAIL(APS_ERR_ARGS, "", "K is NULL");
  *K = 0;
  if (N1 == 0 || N2 == 0) return APS_OK;  // matchFeaturesScratch.m:84-88
  if (!F1 || !F2 || !matches || !metric) APS_FAIL(APS_ERR_ARGS, "", "null pointer argument");
  if (Dbits <= 0) APS_FAIL(APS_ERR_DIM, "", "descriptor width must be positive");
  cudaStream_t s = c->stream;
  const int nb = (Dbits + 7) / 8, nb16 = (nb + 15) / 16 * 16;
  DevBuf<uint8_t> bits[2], packed[2], padded[2], tmp;
  const uint8_t* src[2] = {F1, F2};
  const int64_t cnt[2] = {N1, N2};
  for (int i = 0; i < 2; ++i) {
    APS_TRY(bits[i].alloc((size_t)cnt[i] * Dbits, s));
    APS_TRY(packed[i].alloc((size_t)cnt[i] * nb, s));
    APS_TRY(padded[i].alloc((size_t)cnt[i] * nb16, s));
    APS_TRY(stage_matrix(c, src[i], cnt[i], Dbits, 1, layout, bits[i].p, tmp));
    k_pack_bits01<<<(unsigned)aps_ceil_div(cnt[i] * nb, 256), 256, 0, s>>>(bits[i].p, cnt[i], Dbits, nb, packed[i].p);
    APS_LAUNCHED();
    APS_TRY(pad_rows(s, packed[i].p, cnt[i], nb, nb16, padded[i].p));
  }
  DevBuf<uint32_t> idx2, dm;
  DevBuf<float> d1, d2;
  DevBuf<unsigned long long> best, keys;
  DevBuf<double> dmet;
  DevBuf<int32_t> count;
  APS_TRY(idx2.alloc((size_t)N1, s));
  APS_TRY(d1.alloc((size_t)N1, s));
  APS_TRY(d2.alloc((size_t)N1, s));
  APS_TRY(best.alloc((size_t)N2, s));
  APS_TRY(keys.alloc((size_t)N1 * 2, s));
  APS_TRY(dm.alloc((size_t)N1 * 2, s));
  APS_TRY(dmet.alloc((size_t)N1, s));
  APS_TRY(count.alloc(1, s));
  APS_TRY(hamming2_device(c, padded[0].p, 0, N1, padded[1].p, 0, N2, nb, nb16, idx2.p, d1.p, d2.p));
  APS_TRY(aps_k_pair_filter_unique(s, idx2.p, d1.p, d2.p, N1, N2, 1, /*nBits*/ Dbits, match_threshold, max_ratio, unique,
                                   best.p, keys.p, count.p, dm.p, dmet.p));
  int32_t hk = 0;
  APS_CUDA(cudaMemcpyAsync(&hk, count.p, 4, cudaMemcpyDeviceToHost, s));
  APS_CUDA(cudaStreamSynchronize(s));
  if (hk > 0) {
    APS_CUDA(cudaMemcpyAsync(matches, dm.p, (size_t)hk * 8, cudaMemcpyDeviceToHost, s));
    APS_CUDA(cudaMemcpyAsync(metric, dmet.p, (size_t)hk * 8, cudaMemcpyDeviceToHost, s));
    APS_CUDA(cudaStreamSynchronize(s));
  }
  *K = hk;
  return APS_OK;
}

__global__ void k_gather_pairs(const uint32_t* __restrict__ src_m, const double* __restrict__ src_d,
                               const int64_t* __restrict__ region_off, const int64_t* __restrict__ out_off,
                               uint32_t* __restrict__ rows, double* __restrict__ metric) {
  const int p = blockIdx.x;
  const int64_t a = out_off[p], b = out_off[p + 1], r0 = region_off[p];
  for (int64_t t = threadIdx.x; t < b - a; t += blockDim.x) {
    rows[2 * (a + t)] = src_m[2 * (r0 + t)];
    rows[2 * (a + t) + 1] = src_m[2 * (r0 + t) + 1];
    metric[a + t] = src_d[r0 + t];
  }
}

// One batch of pairs (all using the same descriptor view and engine) through the batched pipeline; results are
// appended to `res`.
static int pairwise_batch(aps_ctx* c, PairwiseSets& ps, const std::vector<PairRef>& pairs, const int64_t* counts, int D,
                          int dtype, bool norm, bool tensor, int dist_metric, double match_threshold, double max_ratio,
                          PairResults& res, const PcaViews* pv) {
  const int np = (int)pairs.size();
  if (np == 0) return APS_OK;
  cudaStream_t s = c->stream;
  if (pv) D = pv->D;
  std::vector<int64_t> eoff(np + 1, 0), boff(np + 1, 0);
  std::vector<int32_t> qoff(np), toff(np), tcnt(np);
  for (int p = 0; p < np; ++p) {
    eoff[p + 1] = eoff[p] + counts[pairs[p].i];
    boff[p + 1] = boff[p] + (pv ? counts[pairs[p].j] : ps.tcnt(pairs[p].j, counts));
    qoff[p] = (int32_t)(pairs[p].qbase >= 0 ? pairs[p].qbase : ps.off[pairs[p].i]);
    toff[p] = (int32_t)(pv ? ps.off[pairs[p].j] : ps.toff(pairs[p].j));   // the train image's rows, or its subset view
    tcnt[p] = (int32_t)(pv ? counts[pairs[p].j] : ps.tcnt(pairs[p].j, counts));
  }
  const int64_t E = eoff[np], B = boff[np];
  DevBuf<int64_t> d_eoff, d_boff;
  DevBuf<int32_t> d_qoff, d_toff, d_tcnt, d_count, fb;
  DevBuf<uint32_t> i2, idx2, matches;
  DevBuf<float> dd, d1, d2;
  DevBuf<unsigned long long> best, keys, winners;
  DevBuf<double> metric;
  APS_TRY(d_eoff.alloc(np + 1, s));
  APS_TRY(d_boff.alloc(np + 1, s));
  APS_TRY(d_qoff.alloc(np, s));
  APS_TRY(d_toff.alloc(np, s));
  APS_TRY(d_tcnt.alloc(np, s));
  APS_TRY(d_count.alloc(np, s));
  APS_TRY(i2.alloc((size_t)E * 2, s));
  APS_TRY(dd.alloc((size_t)E * 2, s));
  APS_TRY(idx2.alloc((size_t)E, s));
  APS_TRY(d1.alloc((size_t)E, s));
  APS_TRY(d2.alloc((size_t)E, s));
  APS_TRY(best.alloc((size_t)B, s));
  APS_TRY(keys.alloc((size_t)E, s));
  APS_TRY(winners.alloc((size_t)E, s));
  APS_TRY(matches.alloc((size_t)E * 2, s));
  APS_TRY(metric.alloc((size_t)E, s));
  APS_CUDA(cudaMemcpyAsync(d_eoff.p, eoff.data(), (np + 1) * 8, cudaMemcpyHostToDevice, s));
  APS_CUDA(cudaMemcpyAsync(d_boff.p, boff.data(), (np + 1) * 8, cudaMemcpyHostToDevice, s));
  APS_CUDA(cudaMemcpyAsync(d_qoff.p, qoff.data(), np * 4, cudaMemcpyHostToDevice, s));
  APS_CUDA(cudaMemcpyAsync(d_toff.p, toff.data(), np * 4, cudaMemcpyHostToDevice, s));
  APS_CUDA(cudaMemcpyAsync(d_tcnt.p, tcnt.data(), np * 4, cudaMemcpyHostToDevice, s));
  aps_pair_tables pt;
  memset(&pt, 0, sizeof pt);
  pt.eoff = d_eoff.p; pt.qoff = d_qoff.p; pt.toff = d_toff.p; pt.tcnt = d_tcnt.p; pt.boff = d_boff.p; pt.npairs = np;
  if (dtype == APS_F32 && ps.subsets() && !pv) {
    pt.vmap = ps.vmap.p;
    pt.vfirst = ps.Freal;
  }

  if (dtype == APS_U8) {
    APS_TRY(aps_k_pairs_hamming2(s, ps.u8pad.p, ps.nb16, eoff, qoff, toff, tcnt, i2.p, dd.p));
    APS_TRY(aps_k_pairs_k2_to_nn(s, pt, E, 1, D, i2.p, dd.p, idx2.p, d1.p, d2.p));
    APS_TRY(aps_k_pairs_filter_unique(s, pt, E, B, idx2.p, d1.p, d2.p, 1, D * 8, match_threshold, max_ratio, best.p,
                                      keys.p, winners.p, d_count.p, matches.p, metric.p));
  } else {
    FloatSet& S = norm ? ps.normset : ps.rawset;
    FloatSide side = S.side();
    TrainView tv = train_view(ps, norm);
    int bias_mode = norm ? 0 : 1;
    const int32_t* flags_dev = S.flags.p;
    const void* q_xh = norm ? (const void*)ps.xh_norm.p : (const void*)ps.xh_raw.p;
    if (pv) {   // 'pca2nn': projected, normalised rows on both sides; cosine scores (scale 1, no bias)
      side.xn = pv->q_xn; side.sq = pv->q_sq; side.invn = pv->q_invn; side.N = pv->qN;
      tv.xn = pv->t_xn; tv.sq = pv->t_sq; tv.xh = pv->t_xh; tv.N = pv->tN; tv.ones = ps.ones.p; tv.colbias = ps.ones.p;
      bias_mode = 0;
      flags_dev = pv->flags;
      q_xh = pv->q_xh;
    }
    c->stats[0] += E;
    if (tensor) {
      c->stats[2] = 2;   // the tensor engine ran for some pair of the call
      std::vector<aps_tc_unit> units;
      for (int p = 0; p < np; ++p) {
        const int64_t nq = eoff[p + 1] - eoff[p];
        for (int64_t b0 = 0; b0 < nq; b0 += 256) {
          aps_tc_unit u;
          u.qrow0 = (int32_t)(qoff[p] + b0);
          u.qend = (int32_t)(qoff[p] + nq);
          u.t0 = toff[p];
          u.t1 = toff[p] + tcnt[p];
          u.out_row = eoff[p] + b0;
          units.push_back(u);
        }
      }
      DevBuf<aps_tc_unit> d_units;
      DevBuf<uint32_t> cidx;
      DevBuf<float> cscore;
      APS_TRY(d_units.alloc(units.size(), s));
      // candidates per (query, train image): k = 2 needs the two best and one witness.  4 = one streaming top-4 list;
      // 3 = branch-free segment epilogue, two sorted lists of three (aps_knn_tc.cu, k_knn_tc<.., 3, 2>)
      // auto: the segment epilogue costs the same for every tile, the streaming one gets cheaper as a sweep goes on
      // (inserts become rare): measured 52 vs 66 ms per batch at 32 tiles per sweep (profiles/r1_ncu_history.txt)
      int64_t tile_steps = 0;
      for (const aps_tc_unit& u : units) tile_steps += ((int64_t)u.t1 - u.t0 + 127) / 128;
      const bool segment_epilogue = c->pairwise_epilogue == 1 ||
                                    (c->pairwise_epilogue < 0 && tile_steps <= 48 * (int64_t)units.size());
      const int KCP = segment_epilogue ? 3 : 4;
      const int nlist = KCP == 3 ? aps_k_knn_tc_tile_mode_stride() / 3 : 1;
      const int cstride = nlist * KCP;
      APS_TRY(cidx.alloc((size_t)E * cstride, s));
      APS_TRY(cscore.alloc((size_t)E * cstride, s));
      APS_TRY(fb.alloc((size_t)E + 1, s));
      APS_CUDA(cudaMemsetAsync(fb.p + E, 0, sizeof(int32_t), s));
      APS_CUDA(cudaMemcpyAsync(d_units.p, units.data(), units.size() * sizeof(aps_tc_unit), cudaMemcpyHostToDevice, s));
      APS_CUDA(cudaStreamSynchronize(s));  // host tables are pageable
      aps_tc_problem tp;
      // fp16 operand rows (built for the screen; |x| <= 2 in this path) when present: 4x smaller operand-rounding
      // term in the proof's eps than bf16, so far fewer rows end in the exact fallback
      const void* xh = q_xh;
      tp.Qb = xh ? (const __nv_bfloat16*)xh : side.xb;
      tp.Tb = xh ? (const __nv_bfloat16*)tv.xh : side.xb_t;
      tp.operand_fp16 = xh ? 1 : 0;
      tp.colscale = xh ? tv.ones : side.colscale_t;
      tp.colbias = xh ? tv.colbias : side.colbias_t;
      tp.tile_bounds = side.tile_bounds; tp.bias = bias_mode;
      tp.Fq_total = side.N; tp.Ft_total = xh ? tv.N : side.N; tp.Dp = (D + 63) / 64 * 64;
      tp.q0 = 0; tp.q1 = 0; tp.t0 = 0; tp.t1 = 0; tp.nslot = 1; tp.kcand = KCP;
      tp.cand_idx = cidx.p; tp.cand_score = cscore.p; tp.dump = nullptr;
      cudaEvent_t ev0 = nullptr, ev1 = nullptr;
      if (c->timing) {
        APS_CUDA(cudaEventCreate(&ev0));
        APS_CUDA(cudaEventCreate(&ev1));
        APS_CUDA(cudaEventRecord(ev0, s));
      }
      APS_TRY(aps_k_knn_tc_units(s, c->sm_count, tp, d_units.p, (int64_t)units.size()));
      if (c->timing) {
        APS_CUDA(cudaEventRecord(ev1, s));
        c->tc_events.push_back(ev0);
        c->tc_events.push_back(ev1);
      }
      aps_pair_tables ptr_ = pt;  // re-rank may skip rows the ratio / threshold test provably rejects
      ptr_.prune = 1;
      ptr_.prune_r2 = max_ratio * max_ratio;
      ptr_.prune_mt = match_threshold;
      ptr_.tile_mode = KCP == 3 ? aps_k_knn_tc_tile_mode_segment() : 0;
      ptr_.operand_fp16 = tp.operand_fp16;
      APS_TRY(aps_k_rerank(s, side.xn, side.sq, side.invn, tv.xn, tv.sq, D, dist_metric, 0, E, 0, nlist, KCP, cidx.p,
                           cscore.p, flags_dev, bias_mode, flags_dev, 2, 0, i2.p, dd.p, fb.p, fb.p + E, &ptr_));
      APS_TRY(aps_k_pair_exact2(s, side.xn, side.sq, tv.xn, tv.sq, D, dist_metric, pt, fb.p, fb.p + E, E, i2.p, dd.p));
      APS_CUDA(cudaMemcpyAsync(c->h_flags + 33, fb.p + E, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    } else {
      if (c->stats[2] == 0) c->stats[2] = 1;
      APS_CUDA(cudaStreamSynchronize(s));
      APS_TRY(aps_k_pair_exact2(s, side.xn, side.sq, tv.xn, tv.sq, D, dist_metric, pt, nullptr, nullptr, E, i2.p, dd.p));
    }
    APS_TRY(aps_k_pairs_k2_to_nn(s, pt, E, 0, 0, i2.p, dd.p, idx2.p, d1.p, d2.p));
    APS_TRY(aps_k_pairs_filter_unique(s, pt, E, B, idx2.p, d1.p, d2.p, 0, 0, match_threshold, max_ratio, best.p, keys.p,
                                      winners.p, d_count.p, matches.p, metric.p));
  }
  // results -> host (regions are compacted on the device first)
  std::vector<int32_t> hc(np);
  APS_CUDA(cudaMemcpyAsync(hc.data(), d_count.p, np * 4, cudaMemcpyDeviceToHost, s));
  APS_CUDA(cudaStreamSynchronize(s));
  if (tensor && dtype == APS_F32) {
    c->stats[1] += c->h_flags[33];
    c->h_flags[32] = (int32_t)c->stats[1];  // aps_ctx_last_stats reports the fallback rows of a tensor search from here
  }
  std::vector<int64_t> outoff(np + 1, 0);
  for (int p = 0; p < np; ++p) outoff[p + 1] = outoff[p] + hc[p];
  const int64_t M = outoff[np];
  // rows and metric of the batch land in ONE pinned staging area (a pageable destination is copied through the
  // driver's bounce buffers at a fraction of the PCIe rate) and are split per pair from there; in device mode they
  // stay in the batch's device buffers
  uint8_t* stage = M > 0 && !res.device ? (uint8_t*)aps_ctx_stage(c, (size_t)M * 16) : nullptr;
  if (M > 0 && !res.device && !stage)
    APS_FAIL(APS_ERR_ALLOC, "", "out of pinned host memory (%lld match rows)", (long long)M);
  const uint32_t* hrows = (const uint32_t*)stage;
  const double* hmet = stage ? (const double*)(stage + (size_t)M * 8) : nullptr;
  if (M > 0) {
    DevBuf<uint32_t> rows_host_mode;
    DevBuf<double> met_host_mode;
    DevBuf<uint32_t>& rows = res.device ? res.d_rows.emplace_back() : rows_host_mode;
    DevBuf<double>& met = res.device ? res.d_met.emplace_back() : met_host_mode;
    DevBuf<int64_t> d_outoff;
    APS_TRY(rows.alloc((size_t)M * 2, s));
    APS_TRY(met.alloc((size_t)M, s));
    APS_TRY(d_outoff.alloc(np + 1, s));
    APS_CUDA(cudaMemcpyAsync(d_outoff.p, outoff.data(), (np + 1) * 8, cudaMemcpyHostToDevice, s));
    k_gather_pairs<<<(unsigned)np, 128, 0, s>>>(matches.p, metric.p, d_eoff.p, d_outoff.p, rows.p, met.p);
    APS_LAUNCHED();
    if (!res.device) {
      APS_CUDA(cudaMemcpyAsync(stage, rows.p, (size_t)M * 8, cudaMemcpyDeviceToHost, s));
      APS_CUDA(cudaMemcpyAsync(stage + (size_t)M * 8, met.p, (size_t)M * 8, cudaMemcpyDeviceToHost, s));
      APS_CUDA(cudaStreamSynchronize(s));
    }
  }
  const int64_t base = res.device ? res.M : (int64_t)res.metric.size();
  if (res.device) {
    res.M += M;
  } else {
    res.rows.insert(res.rows.end(), hrows, hrows + 2 * M);
    res.metric.insert(res.metric.end(), hmet, hmet + M);
  }
  for (int p = 0; p < np; ++p) {
    const size_t o = pairs[p].ordinal;
    res.cnt[o] = hc[p];
    res.at[o] = base + outoff[p];
  }
  return APS_OK;
}

// Stage 1 of the batched pairwise path (aps_pair_screen.cu): every pair of `pairs` is screened on the tensor cores
// with fp16 operands; pairs in which no query row can pass the ratio / threshold test are dropped from the list
// (their cell is empty: zero matches), the others go on to the exact pipeline.
static int pairwise_screen_stage(aps_ctx* c, PairwiseSets& ps, std::vector<PairRef>& pairs, const int64_t* counts, int D,
                                 bool norm, double match_threshold, double max_ratio, const PcaViews* pv) {
  const int np = (int)pairs.size();
  if (np == 0) return APS_OK;
  cudaStream_t s = c->stream;
  if (pv) D = pv->D;
  const int Dp = (D + 63) / 64 * 64;
  FloatSet& S = norm ? ps.normset : ps.rawset;
  const void* xh = pv ? pv->q_xh : (norm ? (const void*)ps.xh_norm.p : (const void*)ps.xh_raw.p);
  const float2* bounds = pv ? pv->bounds : (norm ? ps.bounds_norm.p : ps.bounds_raw.p);
  if (!xh || !bounds) return APS_OK;
  std::vector<int32_t> tab((size_t)np * 5);
  std::vector<int64_t> off2((size_t)(np + 1) * 2, 0);
  int32_t *qoff = tab.data(), *qcnt = qoff + np, *toff = qcnt + np, *tcnt = toff + np, *timg = tcnt + np;
  int64_t *eoff = off2.data(), *uoff = eoff + (np + 1);
  for (int p = 0; p < np; ++p) {
    qoff[p] = (int32_t)(pairs[p].qbase >= 0 ? pairs[p].qbase : ps.off[pairs[p].i]);
    qcnt[p] = (int32_t)counts[pairs[p].i];
    toff[p] = (int32_t)(pv ? ps.off[pairs[p].j] : ps.toff(pairs[p].j));
    tcnt[p] = (int32_t)(pv ? counts[pairs[p].j] : ps.tcnt(pairs[p].j, counts));
    timg[p] = pairs[p].j;
    eoff[p + 1] = eoff[p] + counts[pairs[p].i];
    uoff[p + 1] = uoff[p] + (counts[pairs[p].i] + 255) / 256;
  }
  const int64_t E = eoff[np], U = uoff[np];
  DevBuf<int32_t> d_tab, d_surv;
  DevBuf<int64_t> d_off2;
  DevBuf<aps_tc_unit> d_units;
  DevBuf<uint32_t> scr;
  APS_TRY(d_tab.alloc(tab.size(), s));
  APS_TRY(d_off2.alloc(off2.size(), s));
  APS_TRY(d_surv.alloc((size_t)np, s));
  APS_TRY(d_units.alloc((size_t)U, s));
  APS_TRY(scr.alloc((size_t)E, s));
  APS_CUDA(cudaMemcpyAsync(d_tab.p, tab.data(), tab.size() * 4, cudaMemcpyHostToDevice, s));
  APS_CUDA(cudaMemcpyAsync(d_off2.p, off2.data(), off2.size() * 8, cudaMemcpyHostToDevice, s));
  aps_pair_screen_tables t;
  t.qoff = d_tab.p; t.qcnt = d_tab.p + np; t.toff = d_tab.p + 2 * (size_t)np; t.tcnt = d_tab.p + 3 * (size_t)np;
  t.timg = d_tab.p + 4 * (size_t)np; t.eoff = d_off2.p; t.uoff = d_off2.p + (np + 1); t.npairs = np;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  if (c->timing) {
    APS_CUDA(cudaEventCreate(&ev0));
    APS_CUDA(cudaEventCreate(&ev1));
    APS_CUDA(cudaEventRecord(ev0, s));
  }
  const TrainView tv = train_view(ps, norm);
  APS_TRY(aps_k_pair_screen(s, c->sm_count, xh, pv ? pv->qN : S.N, pv ? pv->t_xh : tv.xh, pv ? pv->tN : tv.N, Dp, t,
                            d_units.p, U, scr.p));
  if (c->timing) {
    APS_CUDA(cudaEventRecord(ev1, s));
    c->tc_events.push_back(ev0);
    c->tc_events.push_back(ev1);
  }
  APS_TRY(aps_k_pair_screen_decide(s, scr.p, pv ? pv->q_sq : S.sq.p, t, bounds, pv ? pv->flags : S.flags.p, Dp,
                                   max_ratio * max_ratio, match_threshold, d_surv.p));
  std::vector<int32_t> surv((size_t)np);
  APS_CUDA(cudaMemcpyAsync(surv.data(), d_surv.p, (size_t)np * 4, cudaMemcpyDeviceToHost, s));
  APS_CUDA(cudaStreamSynchronize(s));   // also covers the pageable host tables above
  std::vector<PairRef> keep;
  for (int p = 0; p < np; ++p)
    if (surv[p] > 0) keep.push_back(pairs[p]);
  c->pair_stats[0] += np;
  c->pair_stats[1] += (int64_t)keep.size();
  c->pair_stats[2] += E;
  c->stats[2] = 2;
  pairs.swap(keep);
  return APS_OK;
}

// staged pairwise pipeline: descriptors resident on the device, prepared once, matched per rank share
struct aps_pplan {
  aps_ctx* c = nullptr;
  int n = 0, D = 0, dtype = 0;
  std::vector<int64_t> counts;
  int64_t F = 0, maxc = 0;
  bool tensor = false, prepared = false;
  int method = APS_METHOD_EXHAUSTIVE;  // aps_pplan_set_method
  int64_t subset = 12000;
  uint64_t seed = 0;
  PairwiseSets ps;
};

extern "C" int aps_pplan_create(aps_ctx* c, const int64_t* counts, int n, int D, int dtype, aps_pplan** out) {
  APS_CTX(c);
  if (!out || n < 0 || (n > 0 && !counts)) APS_FAIL(APS_ERR_ARGS, "", "bad arguments");
  *out = nullptr;
  if (dtype != APS_F32 && dtype != APS_U8) APS_FAIL(APS_ERR_TYPE, "", "descriptors must be single or uint8");
  aps_pplan* p = new (std::nothrow) aps_pplan();
  if (!p) APS_FAIL(APS_ERR_ALLOC, "", "out of host memory");
  p->c = c;
  p->n = n;
  p->D = D;
  p->dtype = dtype;
  p->counts.assign(counts, counts + n);
  for (int i = 0; i < n; ++i) {
    if (counts[i] < 0) {
      delete p;
      APS_FAIL(APS_ERR_ARGS, "", "negative feature count");
    }
    p->F += counts[i];
    if (counts[i] > p->maxc) p->maxc = counts[i];
  }
  if (p->F > 0 && D <= 0) {
    delete p;
    APS_FAIL(APS_ERR_DIM, "", "descriptor dimension must be positive");
  }
  if (p->F >= ((int64_t)1 << 31) - 512) {
    delete p;
    APS_FAIL(APS_ERR_ARGS, "", "more than 2^31 descriptors are not supported");
  }
  p->tensor = dtype == APS_F32 && tc_wanted(c, D, p->maxc, p->maxc * (int64_t)n, 2);
  int rc = pairwise_alloc(c, p->ps, p->counts.data(), n, D, dtype);
  if (rc != APS_OK) {
    delete p;
    return rc;
  }
  *out = p;
  return APS_OK;
}
extern "C" void aps_pplan_destroy(aps_pplan* p) {
  if (!p) return;
  cudaSetDevice(p->c->device);
  delete p;
}
extern "C" int64_t aps_pplan_total(const aps_pplan* p) { return p ? p->F : 0; }
extern "C" void* aps_pplan_desc_device(aps_pplan* p) {
  if (!p) return nullptr;
  return p->dtype == APS_F32 ? (void*)p->ps.rawset.raw.p : (void*)p->ps.u8raw.p;
}
extern "C" int aps_pplan_upload(aps_pplan* p, const void* const* desc, int layout) {
  if (!p) APS_FAIL(APS_ERR_ARGS, "", "plan is NULL");
  APS_CTX(p->c);
  p->prepared = false;
  return pairwise_upload(p->c, p->ps, desc, p->counts.data(), p->n, p->D, p->dtype, layout);
}
extern "C" int aps_pplan_prepare(aps_pplan* p) {
  if (!p) APS_FAIL(APS_ERR_ARGS, "", "plan is NULL");
  APS_CTX(p->c);
  APS_TRY(pairwise_finish(p->c, p->ps, p->counts.data(), p->n, p->D, p->dtype, p->tensor));
  if (p->dtype == APS_F32)
    APS_TRY(pairwise_build_train_view(p->c, p->ps, p->counts.data(), p->n, p->D, p->tensor,
                                      p->method == APS_METHOD_APPROX_SUBSETPDIST2 ? p->subset : 0, p->seed));
  if (p->dtype == APS_F32 && p->method == APS_METHOD_APPROX_PCA2NN)
    APS_TRY(pairwise_build_pca(p->c, p->ps, p->counts.data(), p->n, p->D));
  p->prepared = true;
  return APS_OK;
}

extern "C" int aps_pplan_subset_table(aps_pplan* p, int image, int32_t* out) {
  if (!p || !out || image < 0 || image >= p->n) APS_FAIL(APS_ERR_ARGS, "", "bad arguments");
  APS_CTX(p->c);
  if (!p->prepared || !p->ps.subsets() || p->ps.voff[image] < 0)
    APS_FAIL(APS_ERR_ARGS, "", "image %d has no subset view (prepare() with 'subsetpdist2' and more rows than the subset)", image);
  const int64_t o = p->ps.voff[image] - p->ps.Freal;
  APS_CUDA(cudaMemcpyAsync(out, p->ps.vmap.p + o, (size_t)p->ps.vcnt * 4, cudaMemcpyDeviceToHost, p->c->stream));
  APS_CUDA(cudaStreamSynchronize(p->c->stream));
  return APS_OK;
}

extern "C" int aps_pplan_set_method(aps_pplan* p, int method, int64_t subset, uint64_t seed) {
  if (!p) APS_FAIL(APS_ERR_ARGS, "", "plan is NULL");
  if (method < APS_METHOD_EXHAUSTIVE || method > APS_METHOD_APPROX_PCA2NN)
    APS_FAIL(APS_ERR_METHOD, "", "Select a approximate method");   // matchFeaturesScratch.m:156-157
  if (subset < 1) APS_FAIL(APS_ERR_ARGS, "", "subset must be positive");
  p->method = method;
  p->subset = subset;
  p->seed = seed;
  p->prepared = false;   // the train view depends on the method
  return APS_OK;
}

// Device mode of a pass: the batches' rows and metric joined in batch order into dev.rows / dev.metric (one
// device-to-device copy per batch, the batch buffers released), and the table of the pairs that have rows.
static int pairwise_join_rows(aps_ctx* c, PairResults& res, const std::vector<int64_t>& cell, PairwiseRows& dev) {
  cudaStream_t s = c->stream;
  dev.M = res.M;
  APS_TRY(dev.rows.alloc((size_t)dev.M * 2, s));
  APS_TRY(dev.metric.alloc((size_t)dev.M, s));
  int64_t at = 0;
  for (size_t b = 0; b < res.d_met.size(); ++b) {
    const size_t n = res.d_met[b].n;
    APS_CUDA(cudaMemcpyAsync(dev.rows.p + 2 * at, res.d_rows[b].p, n * 8, cudaMemcpyDeviceToDevice, s));
    APS_CUDA(cudaMemcpyAsync(dev.metric.p + at, res.d_met[b].p, n * 8, cudaMemcpyDeviceToDevice, s));
    at += (int64_t)n;
  }
  res.d_rows.clear();
  res.d_met.clear();
  std::vector<int64_t> src;
  dev.tab.clear();
  for (size_t o = 0; o < res.cnt.size(); ++o)
    if (res.cnt[o] > 0) {
      dev.tab.push_back(cell[o]);
      src.push_back(res.at[o]);
    }
  dev.npairs = (int64_t)src.size();
  for (size_t o = 0; o < res.cnt.size(); ++o)
    if (res.cnt[o] > 0) dev.tab.push_back(res.cnt[o]);
  dev.tab.insert(dev.tab.end(), src.begin(), src.end());
  return APS_OK;
}

// One pass of the pairwise pipeline over an explicit pair list: pairs[o] (ordinal o, pooled image indices, engine) has
// its list written to cell cell[o] of `m` (m->pair_ptr: ncells + 1 entries; cells no pair names stay empty).  Pairs
// with an empty side are skipped (matchFeaturesScratch.m:84-88).  The pairs are grouped by view (raw / normalised,
// :105-110 is a per-pair decision) and engine; tensor groups are screened first, then every group runs in batches of at
// most ENTRY_BUDGET query rows.  Host work is O(pairs + match rows + ncells).  dev != NULL: the lists stay on the
// device instead (pairwise_rows_device), m is not used and host work is O(pairs + batches).
static int pairwise_match_pairs(aps_ctx* c, PairwiseSets& ps, const int64_t* counts, int D, int dtype, int method,
                                double match_threshold, double max_ratio, const std::vector<PairRef>& pairs,
                                const std::vector<int64_t>& cell, int64_t ncells, aps_matchlist* m,
                                PairwiseRows* dev = nullptr) {
  // float descriptors: 1 = (a2 + b2) - 2 G of nearest2SSDExhaustive; 2 = Euclidean search squared afterwards ('kdtree'
  // = exact KD-tree search, :142-148; 'subsetpdist2', :149-155, whose candidate subset is ALL of B while N2 <= subset)
  const bool pca = dtype == APS_F32 && method == APS_METHOD_APPROX_PCA2NN;
  const int metric = (dtype == APS_F32 && method != APS_METHOD_EXHAUSTIVE) ? 2 : 1;
  const size_t NP = pairs.size();
  // groups: [view * 2 + engine], raw before normalised, exact before tensor
  std::vector<PairRef> grp[4];
  for (const PairRef& pr : pairs) {
    if (counts[pr.i] == 0 || counts[pr.j] == 0) continue;  // matchFeaturesScratch.m:84-88
    const bool norm = dtype == APS_F32 && (ps.big[pr.i] || ps.big[pr.j]);  // :105-110 is a per-pair decision
    grp[(norm ? 2 : 0) + (pr.tensor ? 1 : 0)].push_back(pr);
  }
  c->pair_stats[0] = c->pair_stats[1] = c->pair_stats[2] = c->pair_stats[3] = 0;
  int rc = APS_OK;
  const bool dbg_t = getenv("APS_TIMING") != nullptr;
  auto dbg_now = [&]() { cudaStreamSynchronize(c->stream); return std::chrono::steady_clock::now(); };
  auto dbg_t0 = dbg_t ? dbg_now() : std::chrono::steady_clock::time_point();
  if (c->pairwise_screen && !pca)
    for (int g = 1; g < 4 && rc == APS_OK; g += 2)
      rc = pairwise_screen_stage(c, ps, grp[g], counts, D, g >= 2, match_threshold, max_ratio);
  auto dbg_t1 = dbg_t ? dbg_now() : dbg_t0;
  PairResults res;
  res.cnt.assign(NP, 0);
  res.at.assign(NP, 0);
  res.device = dev != nullptr;
  const int64_t ENTRY_BUDGET = (int64_t)1 << 25;  // entries per batch: bounds the candidate buffers to ~2 GB
  for (int g = 0; g < 4 && rc == APS_OK; ++g) {
    const std::vector<PairRef>& gp = grp[g];
    const bool norm = g >= 2, tensor = (g & 1) != 0;
    size_t a = 0;
    while (a < gp.size() && rc == APS_OK) {
      size_t b = a;
      int64_t e = 0;
      while (b < gp.size() && (b == a || e + counts[gp[b].i] <= ENTRY_BUDGET)) e += counts[gp[b++].i];
      std::vector<PairRef> batch(gp.begin() + a, gp.begin() + b);
      if (pca)   // projection with the train image's basis is a per-PAIR operation: screen and match batch by batch
        rc = pairwise_pca_batch(c, ps, batch, counts, D, norm, tensor, match_threshold, max_ratio, res);
      else
        rc = pairwise_batch(c, ps, batch, counts, D, dtype, norm, tensor, metric, match_threshold, max_ratio, res);
      a = b;
    }
  }
  auto dbg_t2 = dbg_t ? dbg_now() : dbg_t0;
  if (rc != APS_OK) return rc;
  if (dev) return pairwise_join_rows(c, res, cell, *dev);
  m->pair_ptr.assign((size_t)ncells + 1, 0);
  for (size_t o = 0; o < NP; ++o) m->pair_ptr[(size_t)cell[o] + 1] = res.cnt[o];
  for (int64_t q = 0; q < ncells; ++q) m->pair_ptr[(size_t)q + 1] += m->pair_ptr[(size_t)q];
  m->total = m->pair_ptr[(size_t)ncells];
  m->rows.resize((size_t)m->total * 2);
  m->metric.resize((size_t)m->total);
  for (size_t o = 0; o < NP; ++o) {
    if (res.cnt[o] == 0) continue;
    const int64_t dst = m->pair_ptr[(size_t)cell[o]], src = res.at[o];
    std::copy(res.rows.begin() + 2 * src, res.rows.begin() + 2 * (src + res.cnt[o]), m->rows.begin() + 2 * dst);
    std::copy(res.metric.begin() + src, res.metric.begin() + src + res.cnt[o], m->metric.begin() + dst);
  }
  if (dbg_t) {
    auto dbg_t3 = dbg_now();
    auto ms = [](auto a, auto b) { return std::chrono::duration<double, std::milli>(b - a).count(); };
    fprintf(stderr, "aps_pplan_match: screen %.2f ms, batches %.2f ms, assemble %.2f ms\n", ms(dbg_t0, dbg_t1), ms(dbg_t1, dbg_t2),
            ms(dbg_t2, dbg_t3));
  }
  return APS_OK;
}

extern "C" int aps_pplan_match(aps_pplan* p, double match_threshold, double max_ratio, int pair_first, int pair_stride,
                               aps_matchlist** out) {
  if (!p || !out) APS_FAIL(APS_ERR_ARGS, "", "bad arguments");
  aps_ctx* c = p->c;
  APS_CTX(c);
  *out = nullptr;
  if (pair_stride < 1 || pair_first < 0 || pair_first >= pair_stride) APS_FAIL(APS_ERR_ARGS, "", "bad pair share");
  const int n = p->n;
  c->stats[0] = c->stats[1] = c->stats[2] = c->stats[3] = 0;
  aps_matchlist* m = new (std::nothrow) aps_matchlist();
  if (!m) APS_FAIL(APS_ERR_ALLOC, "", "out of host memory");
  m->n = n;
  m->has_metric = true;
  const size_t cells = (size_t)n * n;
  m->pair_ptr.assign(cells + 1, 0);
  if (p->F == 0 || n < 2) {
    *out = m;
    return APS_OK;
  }
  if (!p->prepared) {
    delete m;
    APS_FAIL(APS_ERR_ARGS, "", "aps_pplan_prepare() has not run since the last upload");
  }
  // pair list in column-major cell order (featureMatchingPairwise.m:48): j outer, i < j inner; this rank's
  // share = every pair_stride-th pair (the reference's parfor distributes the same list over workers)
  std::vector<PairRef> pairs;
  std::vector<int64_t> cell;
  size_t o = 0;
  for (int j = 0; j < n; ++j)
    for (int i = 0; i < j; ++i, ++o) {
      if ((int)(o % (size_t)pair_stride) != pair_first) continue;
      PairRef pr{i, j, pairs.size()};
      pr.tensor = p->tensor;
      pairs.push_back(pr);
      cell.push_back((int64_t)i + (int64_t)j * n);
    }
  const int rc = pairwise_match_pairs(c, p->ps, p->counts.data(), p->D, p->dtype, p->method, match_threshold, max_ratio,
                                      pairs, cell, (int64_t)cells, m);
  if (rc != APS_OK) {
    delete m;
    return rc;
  }
  *out = m;
  return APS_OK;
}

int feature_matching_pairwise_impl(aps_ctx* c, const void* const* desc, const int64_t* counts, int n, int D, int dtype,
                                   int layout, double match_threshold, double max_ratio, int method, int64_t subset,
                                   uint64_t seed, int pair_first, int pair_stride, aps_matchlist** out, bool dev) {
  APS_CTX(c);
  if (!out) APS_FAIL(APS_ERR_ARGS, "", "out is NULL");
  *out = nullptr;
  if (n < 0 || (n > 0 && !counts) || pair_stride < 1 || pair_first < 0 || pair_first >= pair_stride)
    APS_FAIL(APS_ERR_ARGS, "", "bad arguments");
  aps_pplan* p = nullptr;
  APS_TRY(aps_pplan_create(c, counts, n, D, dtype, &p));
  int rc = aps_pplan_set_method(p, method, subset, seed);
  if (rc == APS_OK && p->F > 0 && n >= 2) {
    if (dev) {  // the pooled device matrix of the set: one copy into the plan
      const cudaError_t e = cudaMemcpyAsync(aps_pplan_desc_device(p), desc[0],
                                            (size_t)p->F * D * (dtype == APS_F32 ? 4 : 1), cudaMemcpyDeviceToDevice,
                                            c->stream);
      if (e != cudaSuccess) {
        aps_set_error(APS_ERR_CUDA, "", "descriptor copy failed: %s", cudaGetErrorString(e));
        rc = APS_ERR_CUDA;
      }
    } else
      rc = aps_pplan_upload(p, desc, layout);
    if (rc == APS_OK) rc = aps_pplan_prepare(p);  // an error here must not reach the pair classification (ps.big)
  }
  if (rc == APS_OK) rc = aps_pplan_match(p, match_threshold, max_ratio, pair_first, pair_stride, out);
  aps_pplan_destroy(p);
  return rc;
}

extern "C" int aps_feature_matching_pairwise(aps_ctx* c, const void* const* desc, const int64_t* counts, int n,
                                             int D, int dtype, int layout, double match_threshold, double max_ratio,
                                             aps_matchlist** out) {
  return feature_matching_pairwise_impl(c, desc, counts, n, D, dtype, layout, match_threshold, max_ratio,
                                        APS_METHOD_EXHAUSTIVE, 12000, 0, 0, 1, out);
}

extern "C" int aps_feature_matching_pairwise_shard(aps_ctx* c, const void* const* desc, const int64_t* counts, int n,
                                                   int D, int dtype, int layout, double match_threshold,
                                                   double max_ratio, int pair_first, int pair_stride,
                                                   aps_matchlist** out) {
  return feature_matching_pairwise_impl(c, desc, counts, n, D, dtype, layout, match_threshold, max_ratio,
                                        APS_METHOD_EXHAUSTIVE, 12000, 0, pair_first, pair_stride, out);
}

// ------------------------------------------------------------------------------------------------
// featureMatchingPairwise over many independent image sets in one call.  The reference runs the pairwise stage once per
// dataset folder and once more per connected component; here all sets share ONE pooled plan (one upload, one K1, one
// train view), one pair list that never crosses a set, and one pass of pairwise_match_pairs -- no host loop over sets
// issues device work, so launches and synchronisations do not depend on nsets.
// dev != NULL: the lists stay on the device in *dev (pairwise_rows_device) and out is not used.  dev_src: desc[i] point
// into one pooled row-major device matrix (pooled_image_ptrs), uploaded with one device-to-device copy.
static int pairwise_sets_pass(aps_ctx* c, int nsets, const int* set_images, const void* const* desc,
                              const int64_t* counts, int nimg, int D, int dtype, int layout, double match_threshold,
                              double max_ratio, int method, int64_t subset, uint64_t seed, aps_matchlist** out,
                              PairwiseRows* dev = nullptr, bool dev_src = false) {
  // per image: its index in its own set (the key of its 'subsetpdist2' subset); per set: its first cell.  Set b's
  // pairs: its own column-major strict-upper-triangle list, on the engine its single-set call chooses (aps_pplan_create)
  std::vector<int32_t> local((size_t)nimg);
  std::vector<int64_t> cell_off((size_t)nsets + 1, 0);
  std::vector<PairRef> pairs;
  std::vector<int64_t> cell;
  bool any_tensor = false;
  for (int b = 0, i0 = 0; b < nsets; i0 += set_images[b++]) {
    const int n = set_images[b];
    int64_t maxc = 0;
    for (int i = 0; i < n; ++i) {
      local[(size_t)i0 + i] = i;
      maxc = counts[i0 + i] > maxc ? counts[i0 + i] : maxc;
    }
    const bool tensor = dtype == APS_F32 && tc_wanted(c, D, maxc, maxc * (int64_t)n, 2);
    for (int j = 0; j < n; ++j)
      for (int i = 0; i < j; ++i) {
        if (counts[i0 + i] == 0 || counts[i0 + j] == 0) continue;  // matchFeaturesScratch.m:84-88
        PairRef pr{i0 + i, i0 + j, pairs.size()};
        pr.tensor = tensor;
        any_tensor |= tensor;
        pairs.push_back(pr);
        cell.push_back(cell_off[b] + i + (int64_t)j * n);
      }
    cell_off[(size_t)b + 1] = cell_off[b] + (int64_t)n * n;
  }
  aps_matchlist pooled;
  pooled.pair_ptr.assign((size_t)cell_off[nsets] + 1, 0);
  if (!pairs.empty()) {
    for (int i = 0; i < nimg; ++i)
      if (counts[i] > 0 && (!desc || !desc[i])) APS_FAIL(APS_ERR_ARGS, "", "descriptor pointer %d is NULL", i);
    PairwiseSets ps;
    APS_TRY(pairwise_alloc(c, ps, counts, nimg, D, dtype));
    const int64_t F = ps.off[nimg];
    DevBuf<int64_t> d_off;
    DevBuf<int32_t> img_of_row;
    if (layout != APS_ROW_MAJOR) {   // the transpose needs each row's image
      APS_TRY(d_off.alloc((size_t)nimg + 1, c->stream));
      APS_TRY(img_of_row.alloc((size_t)F, c->stream));
      APS_CUDA(cudaMemcpyAsync(d_off.p, ps.off.data(), ps.off.size() * 8, cudaMemcpyHostToDevice, c->stream));
      APS_TRY(sets_img_of_row(c->stream, d_off.p, nimg, F, img_of_row.p));
    }
    APS_TRY(sets_upload(c, desc, ps.off, d_off.p, img_of_row.p, D, dtype == APS_F32 ? 4 : 1, layout,
                        dtype == APS_F32 ? (void*)ps.rawset.raw.p : (void*)ps.u8raw.p, dev_src));
    APS_TRY(pairwise_finish(c, ps, counts, nimg, D, dtype, any_tensor));
    if (dtype == APS_F32)
      APS_TRY(pairwise_build_train_view(c, ps, counts, nimg, D, any_tensor,
                                        method == APS_METHOD_APPROX_SUBSETPDIST2 ? subset : 0, seed, local.data()));
    if (dtype == APS_F32 && method == APS_METHOD_APPROX_PCA2NN) APS_TRY(pairwise_build_pca(c, ps, counts, nimg, D));
    APS_TRY(pairwise_match_pairs(c, ps, counts, D, dtype, method, match_threshold, max_ratio, pairs, cell,
                                 cell_off[nsets], &pooled, dev));
  }   // the pass's buffers (ps) are released here: only the lists leave it
  if (dev) {
    dev->cell_off = cell_off;
    return APS_OK;
  }
  // one list per set: cells [cell_off[b], cell_off[b + 1]], rows from pair_ptr[cell_off[b]]
  return sets_split_lists(nsets, pooled.pair_ptr, pooled.rows, &pooled.metric, cell_off, set_images, nullptr, out);
}

// the sets pass with its lists split into out[0 .. nsets), statistics of the call (none on failure)
static int pairwise_sets_lists(aps_ctx* c, int nsets, const int* set_images, const void* const* desc,
                               const int64_t* counts, int nimg, int D, int dtype, int layout, double match_threshold,
                               double max_ratio, int method, int64_t subset, uint64_t seed, bool dev_src,
                               aps_matchlist** out) {
  c->stats[0] = c->stats[1] = c->stats[2] = c->stats[3] = 0;
  c->pair_stats[0] = c->pair_stats[1] = c->pair_stats[2] = c->pair_stats[3] = 0;
  c->h_flags[32] = 0;   // fallback rows of the call's tensor batches (aps_ctx_last_stats)
  const int rc = pairwise_sets_pass(c, nsets, set_images, desc, counts, nimg, D, dtype, layout, match_threshold,
                                    max_ratio, method, subset, seed, out, nullptr, dev_src);
  if (rc != APS_OK)
    for (int b = 0; b < nsets; ++b) {
      aps_matchlist_free(out[b]);
      out[b] = nullptr;
    }
  return rc;
}

extern "C" int aps_feature_matching_pairwise_sets(aps_ctx* c, int nsets, const int* set_images, const void* const* desc,
                                                  const int64_t* counts, int D, int dtype, int layout,
                                                  double match_threshold, double max_ratio, int method, int64_t subset,
                                                  uint64_t seed, aps_matchlist** out) {
  // arguments first (the statuses of the single-set call), then the device
  if (!out) APS_FAIL(APS_ERR_ARGS, "", "out is NULL");
  for (int b = 0; b < nsets; ++b) out[b] = nullptr;
  std::vector<int64_t> img_first;
  APS_TRY(pairwise_sets_args(nsets, set_images, counts, D, dtype, method, subset, img_first));
  const int64_t nimg = img_first[nsets];
  APS_CTX(c);
  if (nsets == 0) return APS_OK;
  if (nsets == 1)  // one set: the single-set call itself
    return feature_matching_pairwise_impl(c, desc, counts, set_images[0], D, dtype, layout, match_threshold, max_ratio,
                                          method, subset, seed, 0, 1, out);
  return pairwise_sets_lists(c, nsets, set_images, desc, counts, (int)nimg, D, dtype, layout, match_threshold,
                             max_ratio, method, subset, seed, false, out);
}

// Device input: the host entry's two paths (one set: the single-set plan; several: the sets pass), each fed from the
// pooled device matrix
extern "C" int aps_feature_matching_pairwise_sets_dev(aps_ctx* c, int nsets, const int* set_images,
                                                      const void* d_pooled, const int64_t* counts, int D, int dtype,
                                                      double match_threshold, double max_ratio, int method,
                                                      int64_t subset, uint64_t seed, void* producer_stream,
                                                      aps_matchlist** out) {
  // the host entry's arguments, then the device pointer, the context and the hand-off
  if (!out) APS_FAIL(APS_ERR_ARGS, "", "out is NULL");
  for (int b = 0; b < nsets; ++b) out[b] = nullptr;
  std::vector<int64_t> img_first;
  APS_TRY(pairwise_sets_args(nsets, set_images, counts, D, dtype, method, subset, img_first));
  const int64_t nimg = img_first[nsets];
  int64_t F = 0;
  for (int64_t g = 0; g < nimg; ++g) F += counts[g];
  APS_TRY(dev_inputs(c, F, d_pooled, nullptr, producer_stream));
  if (nsets == 0) return APS_OK;
  const std::vector<const void*> ptrs = pooled_image_ptrs(d_pooled, counts, nimg, D, dtype == APS_F32 ? 4 : 1);
  if (nsets == 1)  // one set: the single-set call itself
    return feature_matching_pairwise_impl(c, ptrs.data(), counts, set_images[0], D, dtype, APS_ROW_MAJOR,
                                          match_threshold, max_ratio, method, subset, seed, 0, 1, out, true);
  return pairwise_sets_lists(c, nsets, set_images, ptrs.data(), counts, (int)nimg, D, dtype, APS_ROW_MAJOR,
                             match_threshold, max_ratio, method, subset, seed, true, out);
}

int pairwise_sets_args(int nsets, const int* set_images, const int64_t* counts, int D, int dtype, int method,
                       int64_t subset, std::vector<int64_t>& img_first) {
  APS_TRY(sets_image_offsets(nsets, set_images, img_first));
  const int64_t nimg = img_first[nsets];
  if (nimg > 0 && !counts) APS_FAIL(APS_ERR_ARGS, "", "counts is NULL");
  if (dtype != APS_F32 && dtype != APS_U8) APS_FAIL(APS_ERR_TYPE, "", "descriptors must be single or uint8");
  if (method < APS_METHOD_EXHAUSTIVE || method > APS_METHOD_APPROX_PCA2NN)
    APS_FAIL(APS_ERR_METHOD, "", "Select a approximate method");   // matchFeaturesScratch.m:156-157
  if (subset < 1) APS_FAIL(APS_ERR_ARGS, "", "subset must be positive");
  // pooled rows, the subset views included: one plan's limit
  int64_t rows = 0;
  for (int64_t i = 0; i < nimg; ++i) {
    if (counts[i] < 0) APS_FAIL(APS_ERR_ARGS, "", "negative feature count");
    rows += counts[i];
    if (dtype == APS_F32 && method == APS_METHOD_APPROX_SUBSETPDIST2 && counts[i] > subset) rows += subset;
  }
  if (rows > 0 && D <= 0) APS_FAIL(APS_ERR_DIM, "", "descriptor dimension must be positive");
  if (rows >= ((int64_t)1 << 31) - 512)
    APS_FAIL(APS_ERR_ARGS, "", "%lld pooled descriptor rows (subset views included) exceed the limit of 2^31 - 512",
             (long long)rows);
  return APS_OK;
}

int pairwise_rows_device(aps_ctx* c, int nsets, const int* set_images, const void* const* desc, const int64_t* counts,
                         int nimg, int D, int dtype, int layout, double match_threshold, double max_ratio, int method,
                         int64_t subset, uint64_t seed, PairwiseRows& R, bool dev) {
  c->stats[0] = c->stats[1] = c->stats[2] = c->stats[3] = 0;
  c->pair_stats[0] = c->pair_stats[1] = c->pair_stats[2] = c->pair_stats[3] = 0;
  c->h_flags[32] = 0;
  return pairwise_sets_pass(c, nsets, set_images, desc, counts, nimg, D, dtype, layout, match_threshold, max_ratio,
                            method, subset, seed, nullptr, &R, dev);
}
