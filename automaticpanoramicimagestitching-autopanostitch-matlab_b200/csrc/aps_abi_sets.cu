// aps_abi_sets.cu -- featureMatchingGlobal over many independent image sets in one call
// (aps_feature_matching_global_sets, include/apsmatch.h).
//
// The reference runs the whole global pipeline once per dataset folder, and once per connected component; a Python user
// matching a directory of panoramas makes one call per panorama.  Every such call pays fixed costs (allocations, a dozen
// launches, several stream synchronisations), and a small set cannot fill the GPU.  Here all sets share ONE pass:
//   pooled upload (+ one transpose launch for column-major input) -> K1 (two launches: the tensor-path sets' rows, then
//   the others, each with its own flag words) ->
//   float sets the single-set call would search on the tensor path: ONE tcgen05 unit-table launch (every 256-row block
//   of a set against that set's rows, natural row order, columns outside the set masked) -> ONE re-rank + proof (t0 = 0:
//   pooled indices) -> the unproven rows, as a device-side list, to ONE set-restricted K2f launch ->
//   the other sets (binary: K4; float below the tensor size: K2f): ONE group-table launch (up to 8 / 256 query rows of
//   one set against that set's rows only) ->
//   K5a on the pooled records (+ the opt-in mutual check, pooled image ids) -> per-set compaction into sum(n_b^2) cells
//   -> one download, split into nsets lists on the host.
// No host loop over sets; the launch and synchronisation count does not depend on nsets.  Every row's neighbour list is
// the one a search of its set alone returns (re-ranked exactly and proven, or searched exactly; ascending train order,
// ties to the lower index), so the lists are bit-identical to the single-set call's.
#include <algorithm>
#include <climits>
#include <new>
#include <vector>

#include "aps_abi_internal.cuh"

namespace {

// row -> image (upper bound in the pooled offsets): no limit on the number of images
__global__ void k_sets_img_of_row(const int64_t* __restrict__ img_off, int nimg, int64_t F, int32_t* __restrict__ img) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= F) return;
  int lo = 0, hi = nimg;  // last image i with img_off[i] <= r (empty images share their offset with the next one)
  while (hi - lo > 1) {
    const int mid = (lo + hi) / 2;
    if (img_off[mid] <= r) lo = mid;
    else hi = mid;
  }
  img[r] = lo;
}

// column-major image blocks staged one after another (image i at element offset img_off[i] * D) -> pooled row-major
template <class T>
__global__ void k_sets_transpose_in(const T* __restrict__ src, const int32_t* __restrict__ img_of_row,
                                    const int64_t* __restrict__ img_off, int64_t F, int D, T* __restrict__ dst) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= F * D) return;
  const int64_t r = e / D;
  const int c = (int)(e - r * D);
  const int i = img_of_row[r];
  const int64_t b = img_off[i], n = img_off[i + 1] - b;
  dst[e] = src[b * D + (int64_t)c * n + (r - b)];
}

}  // namespace

int sets_img_of_row(cudaStream_t s, const int64_t* d_off, int nimg, int64_t F, int32_t* img) {
  if (F == 0) return APS_OK;
  k_sets_img_of_row<<<(unsigned)aps_ceil_div(F, 256), 256, 0, s>>>(d_off, nimg, F, img);
  APS_LAUNCHED();
  return APS_OK;
}

int sets_upload(aps_ctx* c, const void* const* ptrs, const std::vector<int64_t>& off, const int64_t* d_off,
                const int32_t* img_of_row, int D, int esz, int layout, void* raw) {
  cudaStream_t s = c->stream;
  const int nimg = (int)off.size() - 1;
  const int64_t F = off.back();
  if (F == 0) return APS_OK;
  // row-major images land in place; column-major ones are staged and transposed in one launch
  DevBuf<uint8_t> stage;
  uint8_t* dst = (uint8_t*)raw;
  if (layout != APS_ROW_MAJOR) {
    APS_TRY(stage.alloc((size_t)F * D * esz, s));
    dst = stage.p;
  }
  for (int i = 0; i < nimg; ++i)
    if (off[i + 1] > off[i])
      APS_CUDA(cudaMemcpyAsync(dst + (size_t)off[i] * D * esz, ptrs[i], (size_t)(off[i + 1] - off[i]) * D * esz,
                               cudaMemcpyHostToDevice, s));
  if (layout != APS_ROW_MAJOR) {
    const unsigned grid = (unsigned)aps_ceil_div(F * D, 256);
    if (esz == 4)
      k_sets_transpose_in<float><<<grid, 256, 0, s>>>((const float*)stage.p, img_of_row, d_off, F, D, (float*)raw);
    else
      k_sets_transpose_in<uint8_t><<<grid, 256, 0, s>>>(stage.p, img_of_row, d_off, F, D, (uint8_t*)raw);
    APS_LAUNCHED();   // `stage` is released in stream order
  }
  return APS_OK;
}

namespace {

// rows the tensor pass could not prove -> one K2f group each, searched against its own set's rows (device-side list)
__global__ void k_sets_fallback_groups(const int32_t* __restrict__ fb, const int32_t* __restrict__ nfb,
                                       const int32_t* __restrict__ img_of_row, const int64_t* __restrict__ img_off,
                                       const int32_t* __restrict__ img_set, const int32_t* __restrict__ set_img0,
                                       const int32_t* __restrict__ set_n, int4* __restrict__ groups) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= *nfb) return;
  const int row = fb[i], set = img_set[img_of_row[row]], i0 = set_img0[set];
  groups[i] = make_int4(row, 1, (int)img_off[i0], (int)img_off[i0 + set_n[set]]);
}

// The pooled pass over the sets listed in `sets` (indices into the call's sets).  The first `ntensor` of them are float
// sets the single-set call would search on the tensor path: they occupy rows [0, Ft) of the pooled matrix.
int pooled_pass(aps_ctx* c, const std::vector<int>& sets, int ntensor, const std::vector<int64_t>& img_first,
                const int* set_images, const void* const* desc, const int64_t* counts, int D, int dtype, int layout,
                int k, double ratio, int mutual, aps_matchlist** out) {
  cudaStream_t s = c->stream;
  const int nsets = (int)sets.size();
  // pooled images, offsets and set tables
  std::vector<int64_t> off(1, 0), cell_off(1, 0);
  std::vector<int32_t> img_set, set_img0, set_n;
  std::vector<const void*> ptrs;
  int max_n = 0;
  for (int j = 0; j < nsets; ++j) {
    const int b = sets[j], n = set_images[b];
    set_img0.push_back((int32_t)img_set.size());
    set_n.push_back(n);
    cell_off.push_back(cell_off.back() + (int64_t)n * n);
    max_n = std::max(max_n, n);
    for (int i = 0; i < n; ++i) {
      const int64_t g = img_first[b] + i;
      img_set.push_back(j);
      ptrs.push_back(desc ? desc[g] : nullptr);
      off.push_back(off.back() + counts[g]);
    }
  }
  const int nimg = (int)img_set.size();
  const int64_t F = off.back(), cells = cell_off.back();
  const int64_t Ft = ntensor < nsets ? off[set_img0[ntensor]] : F;  // rows of the tensor-path sets
  std::vector<int64_t> pp((size_t)cells + 1, 0);
  std::vector<uint32_t> rows_h;
  c->h_flags[32] = c->h_flags[34] = c->h_flags[35] = c->h_flags[37] = 0;
  if (F > 0) {
    for (int i = 0; i < nimg; ++i)
      if (off[i + 1] > off[i] && !ptrs[i])
        APS_FAIL(APS_ERR_ARGS, "", "descriptor pointer of image %d is NULL but its count is %lld", i,
                 (long long)(off[i + 1] - off[i]));
    // exact-engine group table over the other sets: the largest sets first (their groups are the longest sweeps)
    const int G = dtype == APS_F32 ? APS_EXACT_GROUP_ROWS : aps_k_knn_hamming_group_rows();
    std::vector<int> order;
    for (int j = ntensor; j < nsets; ++j) order.push_back(j);
    auto rows_of = [&](int j) { return off[set_img0[j] + set_n[j]] - off[set_img0[j]]; };
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return rows_of(a) > rows_of(b); });
    std::vector<int4> groups;
    for (int j : order) {
      const int64_t r0 = off[set_img0[j]], r1 = off[set_img0[j] + set_n[j]];
      for (int64_t q = r0; q < r1; q += G)
        groups.push_back(make_int4((int)q, (int)std::min<int64_t>(G, r1 - q), (int)r0, (int)r1));
    }
    // tensor unit table: every 256-row block of a tensor-path set against that set's rows, one list per row
    const int unit_rows = 2 * aps_k_knn_tc_tile_rows();
    std::vector<aps_tc_unit> units;
    for (int j = 0; j < ntensor; ++j) {
      const int64_t r0 = off[set_img0[j]], r1 = off[set_img0[j] + set_n[j]];
      for (int64_t q = r0; q < r1; q += unit_rows) {
        aps_tc_unit u;
        u.qrow0 = (int32_t)q;
        u.qend = (int32_t)r1;
        u.t0 = (int32_t)r0;
        u.t1 = (int32_t)r1;
        u.out_row = q;
        units.push_back(u);
      }
    }
    const int esz = dtype == APS_F32 ? 4 : 1;
    DevBuf<int64_t> d_off, d_cell_off, dir_counts, pair_counts, pair_ptr, rank;
    DevBuf<int32_t> d_tabs, img_of_row, flags, fb;
    DevBuf<int4> d_groups, fb_groups;
    DevBuf<aps_tc_unit> d_units;
    DevBuf<uint8_t> raw, u8pad, keep;
    DevBuf<float> xn, sq, invn, knn_dist, colscale, colbias, cscore;
    DevBuf<__nv_bfloat16> xb;
    DevBuf<uint32_t> knn_idx, rows, cidx;
    DevBuf<int2> records;
    APS_TRY(d_off.alloc((size_t)nimg + 1, s));
    APS_TRY(d_cell_off.alloc((size_t)nsets + 1, s));
    APS_TRY(d_tabs.alloc((size_t)nimg + 2 * nsets, s));
    APS_TRY(d_groups.alloc(groups.size(), s));
    APS_TRY(d_units.alloc(units.size(), s));
    APS_TRY(img_of_row.alloc((size_t)F, s));
    APS_TRY(raw.alloc((size_t)F * D * esz, s));
    std::vector<int32_t> tabs(img_set);
    tabs.insert(tabs.end(), set_img0.begin(), set_img0.end());
    tabs.insert(tabs.end(), set_n.begin(), set_n.end());
    const int32_t* d_img_set = d_tabs.p;
    const int32_t* d_set_img0 = d_tabs.p + nimg;
    const int32_t* d_set_n = d_tabs.p + nimg + nsets;
    APS_CUDA(cudaMemcpyAsync(d_off.p, off.data(), off.size() * 8, cudaMemcpyHostToDevice, s));
    APS_CUDA(cudaMemcpyAsync(d_cell_off.p, cell_off.data(), cell_off.size() * 8, cudaMemcpyHostToDevice, s));
    APS_CUDA(cudaMemcpyAsync(d_tabs.p, tabs.data(), tabs.size() * 4, cudaMemcpyHostToDevice, s));
    if (!groups.empty())
      APS_CUDA(cudaMemcpyAsync(d_groups.p, groups.data(), groups.size() * sizeof(int4), cudaMemcpyHostToDevice, s));
    if (!units.empty())
      APS_CUDA(cudaMemcpyAsync(d_units.p, units.data(), units.size() * sizeof(aps_tc_unit), cudaMemcpyHostToDevice, s));
    APS_TRY(sets_img_of_row(s, d_off.p, nimg, F, img_of_row.p));
    APS_TRY(sets_upload(c, ptrs.data(), off, d_off.p, img_of_row.p, D, esz, layout, raw.p));
    APS_TRY(knn_idx.alloc((size_t)F * k, s));
    APS_TRY(knn_dist.alloc((size_t)F * k, s));
    if (dtype == APS_F32) {
      const float* X = (const float*)raw.p;
      APS_TRY(xn.alloc((size_t)F * D, s));
      APS_TRY(sq.alloc((size_t)F, s));
      APS_TRY(invn.alloc((size_t)F, s));
      // K1 flag words (exact in fp16, max |sq - 1|, max sq, max |x|) of the tensor-path rows [0, Ft) and, apart, of the
      // other rows: the tensor sets' proof bound comes from their own rows only
      static const int32_t init[16] = {1, 0, 0, 0, 0, 0, 0, 0, 1, 0, 0, 0, 0, 0, 0, 0};
      APS_TRY(flags.alloc(16, s));
      int32_t* flags_t = flags.p;
      int32_t* flags_x = flags.p + 8;
      APS_CUDA(cudaMemcpyAsync(flags.p, init, sizeof init, cudaMemcpyHostToDevice, s));
      // featureMatchingGlobal.m:80-84, the global path's arithmetic (eps inside the sqrt); per row, so the bits are the
      // single-set call's
      if (Ft > 0) APS_TRY(aps_k_prepare_norm(s, X, Ft, D, APS_NORM_GLOBAL, xn.p, sq.p, invn.p, flags_t, 1));
      if (F > Ft)
        APS_TRY(aps_k_prepare_norm(s, X + (size_t)Ft * D, F - Ft, D, APS_NORM_GLOBAL, xn.p + (size_t)Ft * D, sq.p + Ft,
                                   invn.p + Ft, flags_x, 1));
      if (Ft > 0) {
        // tcgen05 candidates of every tensor-path set in ONE unit-table launch (natural row order: a set's rows are
        // contiguous, columns outside its range are masked), exact re-rank + completeness proof, unproven rows to K2f
        const int Dp = (D + 63) / 64 * 64;
        const int kcand = k <= 5 ? 8 : 16;
        APS_TRY(xb.alloc((size_t)Ft * Dp, s));
        APS_TRY(colscale.alloc((size_t)Ft + 256, s));
        APS_TRY(colbias.alloc((size_t)Ft + 256, s));
        APS_TRY(aps_k_prepare_operands(s, X, xn.p, sq.p, invn.p, Ft, D, Dp, flags_t, /*bias_mode*/ 0, xb.p, colscale.p,
                                       colbias.p, 1));
        APS_TRY(cidx.alloc((size_t)Ft * kcand, s));
        APS_TRY(cscore.alloc((size_t)Ft * kcand, s));
        aps_tc_problem tp;
        memset(&tp, 0, sizeof tp);
        tp.Qb = xb.p;
        tp.Tb = xb.p;
        tp.colscale = colscale.p;
        tp.colbias = colbias.p;
        tp.bias = 0;
        tp.Fq_total = Ft;
        tp.Ft_total = Ft;
        tp.Dp = Dp;
        tp.nslot = 1;
        tp.kcand = kcand;
        tp.cand_idx = cidx.p;
        tp.cand_score = cscore.p;
        tp.operand_fp16 = 2;  // fp16 operands, flags[0] tells whether they are exact (as aps_gplan_create)
        APS_TRY(aps_k_knn_tc_units(s, c->sm_count, tp, d_units.p, (int64_t)units.size()));
        APS_TRY(fb.alloc((size_t)Ft + 1, s));
        APS_CUDA(cudaMemsetAsync(fb.p + Ft, 0, sizeof(int32_t), s));
        aps_pair_tables gpt;
        memset(&gpt, 0, sizeof gpt);
        gpt.operand_fp16 = tp.operand_fp16;
        APS_TRY(aps_k_rerank(s, xn.p, sq.p, invn.p, xn.p, sq.p, D, /*metric*/ 0, 0, Ft, /*t0*/ 0, /*nseg*/ 1, kcand,
                             cidx.p, cscore.p, flags_t, 0, flags_t, k, 0, knn_idx.p, knn_dist.p, fb.p, fb.p + Ft, &gpt));
        APS_TRY(fb_groups.alloc((size_t)Ft, s));
        k_sets_fallback_groups<<<(unsigned)aps_ceil_div(Ft, 256), 256, 0, s>>>(fb.p, fb.p + Ft, img_of_row.p, d_off.p,
                                                                               d_img_set, d_set_img0, d_set_n,
                                                                               fb_groups.p);
        APS_LAUNCHED();
        APS_TRY(aps_k_knn_exact_groups(s, xn.p, fb_groups.p, Ft, fb.p + Ft, D, k, knn_idx.p, knn_dist.p));
        APS_CUDA(cudaMemcpyAsync(c->h_flags + 32, fb.p + Ft, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
        APS_CUDA(cudaMemcpyAsync(c->h_flags + 35, flags_t, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
      }
      if (F > Ft) {
        APS_TRY(aps_k_knn_exact_groups(s, xn.p, d_groups.p, (int64_t)groups.size(), nullptr, D, k, knn_idx.p,
                                       knn_dist.p));
        APS_CUDA(cudaMemcpyAsync(c->h_flags + 37, flags_x, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
      }
    } else {
      const int nb16 = (D + 15) / 16 * 16;
      APS_TRY(u8pad.alloc((size_t)F * nb16, s));
      APS_TRY(pad_rows(s, raw.p, F, D, nb16, u8pad.p));
      APS_TRY(aps_k_knn_hamming_groups(s, u8pad.p, d_groups.p, (int64_t)groups.size(), nb16, k, knn_idx.p,
                                       knn_dist.p));
    }
    // K5a on the pooled records, the opt-in cross-check, per-set compaction
    APS_TRY(records.alloc((size_t)F, s));
    APS_TRY(aps_k_global_filter(s, knn_idx.p, knn_dist.p, k, 0, F, img_of_row.p, d_off.p, (float)ratio, records.p));
    if (mutual) {
      APS_TRY(keep.alloc((size_t)F, s));
      APS_TRY(aps_k_records_mutual(s, records.p, img_of_row.p, d_off.p, F, keep.p));
    }
    APS_TRY(dir_counts.alloc((size_t)cells, s));
    APS_TRY(pair_counts.alloc((size_t)cells, s));
    APS_TRY(pair_ptr.alloc((size_t)cells + 1, s));
    APS_TRY(rank.alloc((size_t)F, s));
    APS_TRY(rows.alloc((size_t)F * 2, s));
    APS_TRY(aps_k_global_compact_sets(s, records.p, img_of_row.p, d_off.p, nimg, F, d_img_set, d_set_img0, d_set_n,
                                      d_cell_off.p, nsets, max_n, cells, dir_counts.p, pair_counts.p, pair_ptr.p,
                                      rank.p, rows.p));
    APS_CUDA(cudaMemcpyAsync(pp.data(), pair_ptr.p, pp.size() * 8, cudaMemcpyDeviceToHost, s));
    APS_CUDA(cudaStreamSynchronize(s));
    rows_h.resize((size_t)pp[cells] * 2);
    if (pp[cells] > 0) {
      APS_CUDA(cudaMemcpyAsync(rows_h.data(), rows.p, rows_h.size() * 4, cudaMemcpyDeviceToHost, s));
      APS_CUDA(cudaStreamSynchronize(s));
    }
  }
  // split into one list per set (cells of set j: [cell_off[j], cell_off[j + 1]], rows from pp[cell_off[j]])
  for (int j = 0; j < nsets; ++j) {
    aps_matchlist* m = new (std::nothrow) aps_matchlist();
    if (!m) APS_FAIL(APS_ERR_ALLOC, "", "out of host memory");
    out[sets[j]] = m;
    m->n = set_n[j];
    const int64_t c0 = cell_off[j], c1 = cell_off[j + 1], r0 = pp[c0];
    m->pair_ptr.resize((size_t)(c1 - c0) + 1);
    for (int64_t cc = c0; cc <= c1; ++cc) m->pair_ptr[(size_t)(cc - c0)] = pp[cc] - r0;
    m->total = pp[c1] - r0;
    m->rows.assign(rows_h.begin() + 2 * r0, rows_h.begin() + 2 * pp[c1]);
  }
  // statistics of the call, as the single-set call reports them: rows searched; the engine (tcgen05 when any set took
  // the tensor path); rows its proof left to K2f (no second tensor pass here: first-pass unproven == fallback rows);
  // operands exact for every float row
  c->stats[0] = F;
  c->stats[2] = Ft > 0 ? 2 : (F > 0 ? 1 : 0);
  c->stats[1] = Ft > 0 ? c->h_flags[32] : 0;
  c->h_flags[34] = c->h_flags[32];
  c->stats[3] = dtype == APS_F32 && F > 0 && (Ft == 0 || c->h_flags[35]) && (F == Ft || c->h_flags[37]);
  c->h_flags[36] = 0;
  return APS_OK;
}

}  // namespace

extern "C" int aps_feature_matching_global_sets(aps_ctx* c, int nsets, const int* set_images, const void* const* desc,
                                                const int64_t* counts, int D, int dtype, int layout, int k,
                                                double ratio, int use_bf, int mutual, aps_matchlist** out) {
  (void)use_bf;
  // arguments first (the ids of aps_feature_matching_global), then the device
  if (nsets < 0) APS_FAIL(APS_ERR_ARGS, "", "nsets must be >= 0 (got %d)", nsets);
  if (!out) APS_FAIL(APS_ERR_ARGS, "", "out is NULL");
  if (nsets > 0 && !set_images) APS_FAIL(APS_ERR_ARGS, "", "set_images is NULL");
  for (int b = 0; b < nsets; ++b) out[b] = nullptr;
  std::vector<int64_t> img_first((size_t)nsets + 1, 0);
  for (int b = 0; b < nsets; ++b) {
    if (set_images[b] < 0) APS_FAIL(APS_ERR_ARGS, "", "set %d has a negative image count", b);
    img_first[b + 1] = img_first[b] + set_images[b];
  }
  const int64_t nimg = img_first[nsets];
  if (nimg > INT_MAX) APS_FAIL(APS_ERR_ARGS, "", "too many images");
  if (nimg > 0 && !counts) APS_FAIL(APS_ERR_ARGS, "", "counts is NULL");
  std::vector<int64_t> set_rows((size_t)nsets, 0);
  int64_t F = 0;
  for (int b = 0; b < nsets; ++b)
    for (int64_t i = img_first[b]; i < img_first[b + 1]; ++i) {
      if (counts[i] < 0) APS_FAIL(APS_ERR_ARGS, "", "negative feature count");
      set_rows[b] += counts[i];
      F += counts[i];
    }
  if (dtype != APS_F32 && dtype != APS_U8)
    APS_FAIL(APS_ERR_TYPE, "flann_knn:type", "Descriptors must be single (float) or uint8 (binary)");
  if (k <= 0) APS_FAIL(APS_ERR_K, "flann_knn:k", "k must be > 0");
  if (k > APS_MAX_K) APS_FAIL(APS_ERR_K, "flann_knn:k", "k must be <= %d in this implementation", APS_MAX_K);
  if (F > 0 && D <= 0) APS_FAIL(APS_ERR_DIM, "flann_knn:dim", "descriptor dimension must be positive");
  if (F >= ((int64_t)1 << 31) - 1) APS_FAIL(APS_ERR_ARGS, "", "more than 2^31 descriptors are not supported");
  APS_CTX(c);
  if (nsets == 0) return APS_OK;
  if (nsets == 1)  // one set: the single-set call itself
    return feature_matching_global_impl(c, desc, counts, set_images[0], D, dtype, layout, k, ratio, mutual, out);

  // one pass for every set: float sets the single-set call would search on the tensor path first (rows [0, Ft) of the
  // pooled matrix, one tcgen05 unit-table launch), then the sets it would search with the exact engines
  std::vector<int> order, rest;
  for (int b = 0; b < nsets; ++b)
    (dtype == APS_F32 && set_rows[b] > 0 && tc_wanted(c, D, set_rows[b], set_rows[b], k) ? order : rest).push_back(b);
  const int ntensor = (int)order.size();
  order.insert(order.end(), rest.begin(), rest.end());
  const int rc = pooled_pass(c, order, ntensor, img_first, set_images, desc, counts, D, dtype, layout, k, ratio, mutual,
                             out);
  if (rc != APS_OK)
    for (int b = 0; b < nsets; ++b) {
      aps_matchlist_free(out[b]);
      out[b] = nullptr;
    }
  return rc;
}
