// aps_global_image_matching.cu -- featureMatchingGlobal or featureMatchingPairwise followed by imageMatching in one
// call (aps_global_image_matching_sets, aps_pairwise_image_matching_sets, include/apsmatch.h).
//
// The reference calls featureMatchingGlobal (input.matchFeaturesPairwise = 0) or featureMatchingPairwise (= 1) and then
// imageMatching on the same image set.  As two calls, the match lists travel to the host and back: downloaded and split
// per set, turned into cells, counted and packed again on the host, uploaded again.  Here they stay on the device:
//   global pass (aps_feature_matching_global_sets up to its compaction: pair_counts, pair_ptr, rows in pass order), or
//   pairwise pass (aps_feature_matching_pairwise_sets with each batch's rows kept on the device) -> k_scatter_counts
//   (pair_counts) -> k_scan_counts (pair_ptr) -> k_place_rows (rows and metric in cell order), then the shared tail:
//   K6 partner selection directly on pair_counts (k_select_rows / k_select_sym / k_select_compact) ->
//   k_candidate_tables (images, key, cell and putative count of every candidate pair) -> k_scan_counts (pt_ptr) ->
//   k_pack_rows (the candidate pairs' match rows, packed) -> the only synchronisation of the tail: number of pairs and
//   of correspondences -> the gather + RANSAC chunks of aps_image_matching_sets -> k_scan_counts (allMatches offsets) ->
//   k_all_matches (rows with the inlier flag set, accepted pairs only) -> one download, reordered into the caller's set
//   order on the host.
// A set's candidate pairs are keyed by their index in that set's own list, so pass order changes nothing: every output
// is the two-call chain's, bit for bit.  The *_dev entries take the descriptors and keypoints from device memory: the
// passes copy the pooled descriptors device-to-device where they upload, and match_lists copies float64 keypoints or
// widens float32 ones on the device (k_widen_keypoints) where it uploads; the rest is the same code.
#include <climits>
#include <new>
#include <vector>

#include "aps_abi_internal.cuh"

struct aps_image_matches {
  int nsets = 0;
  std::vector<int64_t> set_pair_ptr, pairs_lin, pt_ptr, match_ptr;
  std::vector<uint32_t> match_rows;
  std::vector<double> models, models_inv;
  std::vector<int32_t> n_inliers, draws_used;
  std::vector<uint8_t> accepted;
  std::vector<aps_matchlist*> lists;  // empty unless the call asked for them
  ~aps_image_matches() {
    for (aps_matchlist* m : lists) aps_matchlist_free(m);
  }
};

namespace {

// the pass position whose range [ptr[j], ptr[j + 1]) holds x (last j < n with ptr[j] <= x)
__device__ __forceinline__ int64_t last_le(const int64_t* __restrict__ ptr, int64_t n, int64_t x) {
  int64_t lo = 0, hi = n;
  while (hi - lo > 1) {
    const int64_t mid = (lo + hi) >> 1;
    if (ptr[mid] <= x) lo = mid;
    else hi = mid;
  }
  return lo;
}

// Set tables of the pass, one int64 array: [set_img (nsets + 1) | cell_off (nsets + 1) | img0 (nsets) | n (nsets) |
// img_off (images + 1)].  set_img and cell_off follow the pass order, img0 is each pass position's first image in the
// caller's pooled order (that of img_off and the keypoints).
struct PassTables {
  const int64_t* set_img;
  const int64_t* cell_off;
  const int64_t* img0;
  const int64_t* n;
};

// One thread per candidate pair slot p < cap (pairs past set_pair_ptr[nsets] get a zero count): the pair's set j, its
// cell, its two images in the caller's pooled order, its sample key (index in its own set's list) and its putative
// count (imageMatching.m:76, putativeCount = size(matchesAll{i,j}, 1)).
__global__ void k_candidate_tables(const int64_t* __restrict__ pairs_lin, const int64_t* __restrict__ set_pair_ptr,
                                   int nsets, int64_t cap, PassTables t, const int64_t* __restrict__ pair_ptr,
                                   int64_t* __restrict__ cell, int32_t* __restrict__ ii, int32_t* __restrict__ jj,
                                   int64_t* __restrict__ keys, int64_t* __restrict__ cnt) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= cap) return;
  if (p >= set_pair_ptr[nsets]) {
    cnt[p] = 0;
    return;
  }
  const int64_t j = last_le(set_pair_ptr, nsets, p);
  const int64_t lin = pairs_lin[p], n = t.n[j], c = t.cell_off[j] + lin;
  cell[p] = c;
  ii[p] = (int32_t)(t.img0[j] + lin % n);
  jj[p] = (int32_t)(t.img0[j] + lin / n);
  keys[p] = p - set_pair_ptr[j];
  cnt[p] = pair_ptr[c + 1] - pair_ptr[c];
}

struct CountOf {  // count of entry i: a table
  const int64_t* c;
  __device__ int64_t operator()(int64_t i) const { return c[i]; }
};
struct AcceptedInliers {  // rows allMatches keeps of pair i: its inliers when accepted (imageMatching.m:147-148)
  const uint8_t* acc;
  const int32_t* ni;
  __device__ int64_t operator()(int64_t i) const { return acc[i] ? ni[i] : 0; }
};

// exclusive scan of n counts into out[0..n] (out[n] = the sum, also written to *total when total != NULL); one CTA,
// each thread a contiguous range
template <class Count>
__global__ void __launch_bounds__(1024) k_scan_counts(Count cnt, int64_t n, int64_t* __restrict__ out,
                                                      int64_t* __restrict__ total) {
  __shared__ int64_t s_part[1024];
  const int tid = threadIdx.x, nt = blockDim.x;
  const int64_t per = (n + nt - 1) / nt;
  const int64_t c0 = min(n, tid * per), c1 = min(n, c0 + per);
  int64_t sum = 0;
  for (int64_t i = c0; i < c1; ++i) sum += cnt(i);
  s_part[tid] = sum;
  __syncthreads();
  if (tid == 0) {
    int64_t run = 0;
    for (int t = 0; t < nt; ++t) {
      const int64_t v = s_part[t];
      s_part[t] = run;
      run += v;
    }
    out[n] = run;
    if (total) *total = run;
  }
  __syncthreads();
  int64_t run = s_part[tid];
  for (int64_t i = c0; i < c1; ++i) {
    out[i] = run;
    run += cnt(i);
  }
}

// The candidate pairs' match rows, packed in pair order (what aps_image_matching_sets builds on the host): output row
// r < pt_ptr[np] belongs to the pair p whose range holds it and copies row r - pt_ptr[p] of that pair's cell.
__global__ void k_pack_rows(const int64_t* __restrict__ set_pair_ptr, int nsets, const int64_t* __restrict__ pt_ptr,
                            const int64_t* __restrict__ cell, const int64_t* __restrict__ pair_ptr,
                            const uint2* __restrict__ rows, uint2* __restrict__ packed) {
  const int64_t np = set_pair_ptr[nsets], total = pt_ptr[np];
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < total; r += (int64_t)gridDim.x * blockDim.x) {
    const int64_t p = last_le(pt_ptr, np, r);
    packed[r] = rows[pair_ptr[cell[p]] + (r - pt_ptr[p])];
  }
}

// allMatches{ii,jj} = matches(inliers,:) (imageMatching.m:148) of every accepted pair: one CTA per pair keeps the
// flagged rows in their order, at out_ptr[pair].  k_ransac_final counts n_inliers over the same flags, so the rows fill
// [out_ptr[pair], out_ptr[pair + 1]) exactly.
__global__ void __launch_bounds__(256) k_all_matches(const int64_t* __restrict__ pt_ptr, const uint2* __restrict__ rows,
                                                     const uint8_t* __restrict__ inl, const int64_t* __restrict__ out_ptr,
                                                     uint2* __restrict__ out) {
  __shared__ int warp_cnt[8];
  const int64_t pair = blockIdx.x;
  const int64_t o = pt_ptr[pair], n = pt_ptr[pair + 1] - o, end = out_ptr[pair + 1];
  int64_t base = out_ptr[pair];
  if (base == end) return;  // rejected, or nothing to keep (uniform over the CTA)
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
  for (int64_t r0 = 0; r0 < n; r0 += blockDim.x) {
    const int64_t r = r0 + threadIdx.x;
    const bool keep = r < n && inl[o + r];
    const unsigned bal = __ballot_sync(0xffffffffu, keep);
    if (lane == 0) warp_cnt[w] = __popc(bal);
    __syncthreads();
    int before = 0, tot = 0;
    for (int k = 0; k < nw; ++k) {
      before += k < w ? warp_cnt[k] : 0;
      tot += warp_cnt[k];
    }
    const int64_t pos = base + before + __popc(bal & ((1u << lane) - 1u));
    if (keep && pos < end) out[pos] = rows[o + r];
    base += tot;
    __syncthreads();
  }
}

// pair_counts[cell[q]] = count[q] for every pair q with rows of a pairwise pass (PairwiseRows::tab); the other cells
// keep the zero of a memset
__global__ void k_scatter_counts(const int64_t* __restrict__ tab, int64_t np, int64_t* __restrict__ pair_counts) {
  const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (q < np) pair_counts[tab[q]] = tab[np + q];
}

// One CTA per pair with rows of a pairwise pass: its rows (and metric, when met != NULL) from batch order to its cell's
// place pair_ptr[cell] of the cell-ordered lists
__global__ void __launch_bounds__(128) k_place_rows(const int64_t* __restrict__ tab, int64_t np,
                                                    const int64_t* __restrict__ pair_ptr,
                                                    const uint2* __restrict__ src_rows,
                                                    const double* __restrict__ src_met, uint2* __restrict__ rows,
                                                    double* __restrict__ met) {
  const int64_t q = blockIdx.x;
  const int64_t n = tab[np + q], s0 = tab[2 * np + q], d0 = pair_ptr[tab[q]];
  for (int64_t t = threadIdx.x; t < n; t += blockDim.x) {
    rows[d0 + t] = src_rows[s0 + t];
    if (met) met[d0 + t] = src_met[s0 + t];
  }
}

// float32 keypoints -> double2, exactly (every float is a double): one thread per keypoint, two scalar loads, so the
// caller's pointer needs no more than float alignment
__global__ void k_widen_keypoints(const float* __restrict__ src, int64_t n, double2* __restrict__ dst) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = make_double2((double)src[2 * i], (double)src[2 * i + 1]);
}

// Where the pooled [F x 2] keypoints come from: host float64 (the host entries), or device memory (the *_dev entries)
// of aps_kp_dtype `dtype`
struct KeypointSource {
  const void* p;
  bool dev;
  int dtype;
};

// candidate pairs a set can have at most: every image marks at most min(m, n - 1) partners (imageMatching.m:86-91)
int64_t pair_bound(const std::vector<int>& ns, int m) {
  int64_t cap = 0;
  for (int n : ns) {
    const int64_t take = n > 1 ? (m < 0 ? 0 : (m < n - 1 ? m : n - 1)) : 0;
    cap += std::min<int64_t>((int64_t)n * (n - 1) / 2, (int64_t)n * take);
  }
  return cap;
}

// The caller's set b sits at pass position pos[b]; its pass pairs are spp[pos[b]] .. spp[pos[b] + 1].  Every per-pair
// array is copied set after set in the caller's order; pt_ptr / match_ptr are rebuilt from the counts.
void reorder(const std::vector<int>& order, const std::vector<int64_t>& spp, const int64_t* lin, const int64_t* pt,
             const int64_t* am, const uint32_t* am_rows, const double* models, const double* minv, const int32_t* ni,
             const uint8_t* acc, const int32_t* used, aps_image_matches* r) {
  const int nsets = (int)order.size();
  const int64_t P = spp[nsets];
  std::vector<int> pos((size_t)nsets);
  for (int j = 0; j < nsets; ++j) pos[order[j]] = j;
  r->set_pair_ptr.assign((size_t)nsets + 1, 0);
  r->pairs_lin.resize((size_t)P);
  r->pt_ptr.assign((size_t)P + 1, 0);
  r->match_ptr.assign((size_t)P + 1, 0);
  r->match_rows.resize((size_t)(2 * am[P]));
  r->models.resize((size_t)P * 9);
  r->models_inv.resize((size_t)P * 9);
  r->n_inliers.resize((size_t)P);
  r->accepted.resize((size_t)P);
  r->draws_used.resize((size_t)P);
  int64_t q = 0;
  for (int b = 0; b < nsets; ++b) {
    const int64_t p0 = spp[pos[b]], p1 = spp[pos[b] + 1];
    std::copy(am_rows + 2 * am[p0], am_rows + 2 * am[p1], r->match_rows.begin() + 2 * r->match_ptr[q]);
    for (int64_t p = p0; p < p1; ++p, ++q) {
      r->pairs_lin[q] = lin[p];
      r->pt_ptr[q + 1] = r->pt_ptr[q] + (pt[p + 1] - pt[p]);
      r->match_ptr[q + 1] = r->match_ptr[q] + (am[p + 1] - am[p]);
      std::copy(models + 9 * p, models + 9 * p + 9, r->models.begin() + 9 * q);
      std::copy(minv + 9 * p, minv + 9 * p + 9, r->models_inv.begin() + 9 * q);
      r->n_inliers[q] = ni[p];
      r->accepted[q] = acc[p];
      r->draws_used[q] = used[p];
    }
    r->set_pair_ptr[b + 1] = q;
  }
}

// imageMatching of every set on lists L that are on the device (both entries): partner selection, candidate tables,
// packed rows, RANSAC, allMatches and the download into r.  F: pooled keypoint rows; row_bound: a bound on the rows of
// L's lists (sizes the packed correspondences).  With want_lists, r->lists are L's lists (with L.metric when set).
int match_lists(aps_ctx* c, int nsets, const int* set_images, const std::vector<int64_t>& img_first,
                const int64_t* counts, int64_t F, const KeypointSource& keypoints, const GlobalLists& L, int64_t row_bound,
                int m, double max_distance, double confidence, int max_trials, uint64_t seed, int want_lists,
                aps_image_matches* r) {
  cudaStream_t s = c->stream;
  const int G = (int)img_first[nsets];
  const std::vector<int>& order = L.order;
  const int64_t cells = L.cell_off.back();
  std::vector<int> ns;
  for (int b : order) ns.push_back(set_images[b]);
  const int64_t cap = pair_bound(ns, m);
  // set tables (PassTables layout) and the caller's image offsets, one upload
  const size_t nt = (size_t)nsets + 1;
  std::vector<int64_t> tab(2 * nt + 2 * (size_t)nsets + (size_t)G + 1, 0);
  for (int j = 0; j < nsets; ++j) {
    tab[j + 1] = tab[j] + ns[j];
    tab[nt + j + 1] = L.cell_off[j + 1];
    tab[2 * nt + j] = img_first[order[j]];
    tab[2 * nt + nsets + j] = ns[j];
  }
  int64_t* img_off = tab.data() + 2 * nt + 2 * nsets;
  for (int g = 0; g < G; ++g) img_off[g + 1] = img_off[g] + counts[g];
  DevBuf<int64_t> dtab, sel, lin, cell, keys, cnt, pt, am;
  DevBuf<int32_t> ii, jj, ni, used;
  DevBuf<uint8_t> cand, acc, inl;
  DevBuf<uint32_t> packed, am_rows;
  DevBuf<double2> kp;
  DevBuf<double> models, minv;
  APS_TRY(dtab.alloc(tab.size(), s));
  APS_CUDA(cudaMemcpyAsync(dtab.p, tab.data(), tab.size() * 8, cudaMemcpyHostToDevice, s));
  const PassTables t{dtab.p, dtab.p + nt, dtab.p + 2 * nt, dtab.p + 2 * nt + nsets};
  const int64_t* d_img_off = dtab.p + 2 * nt + 2 * nsets;
  if (F > 0) {
    APS_TRY(kp.alloc((size_t)F, s));
    if (!keypoints.dev) {
      APS_CUDA(cudaMemcpyAsync(kp.p, keypoints.p, (size_t)F * 16, cudaMemcpyHostToDevice, s));
    } else if (keypoints.dtype == APS_KP_F64) {
      APS_CUDA(cudaMemcpyAsync(kp.p, keypoints.p, (size_t)F * 16, cudaMemcpyDeviceToDevice, s));
    } else {
      k_widen_keypoints<<<(unsigned)aps_ceil_div(F, 256), 256, 0, s>>>((const float*)keypoints.p, F, kp.p);
      APS_LAUNCHED();
    }
  }
  // K6 on the device counts, find() per set: sel = [set_pair_ptr (nsets + 1) | correspondences], pairs_lin in lin
  APS_TRY(sel.alloc(nt + 1, s));
  APS_TRY(lin.alloc((size_t)(cap > 0 ? cap : 1), s));
  APS_TRY(cand.alloc((size_t)(cells > 0 ? cells : 1), s));
  APS_TRY(aps_k_select_partners_sets(s, L.pair_counts, G, cells, t.set_img, t.cell_off, nsets, m, cand.p));
  APS_TRY(aps_k_select_compact(s, cand.p, cells, t.cell_off, nsets, lin.p, sel.p));
  // candidate-pair tables, pt_ptr and the packed rows
  APS_TRY(cell.alloc((size_t)cap, s));
  APS_TRY(ii.alloc((size_t)cap, s));
  APS_TRY(jj.alloc((size_t)cap, s));
  APS_TRY(keys.alloc((size_t)cap, s));
  APS_TRY(cnt.alloc((size_t)cap, s));
  APS_TRY(pt.alloc((size_t)cap + 1, s));
  APS_TRY(packed.alloc((size_t)(row_bound > 0 ? 2 * row_bound : 2), s));
  if (cap > 0) {
    k_candidate_tables<<<(unsigned)aps_ceil_div(cap, 256), 256, 0, s>>>(lin.p, sel.p, nsets, cap, t, L.pair_ptr,
                                                                         cell.p, ii.p, jj.p, keys.p, cnt.p);
    APS_LAUNCHED();
  }
  k_scan_counts<<<1, 1024, 0, s>>>(CountOf{cnt.p}, cap, pt.p, sel.p + nt);
  APS_LAUNCHED();
  if (row_bound > 0 && cap > 0) {
    k_pack_rows<<<(unsigned)aps_min64(aps_ceil_div(row_bound, 256), 8 * (int64_t)c->sm_count), 256, 0, s>>>(
        sel.p, nsets, pt.p, cell.p, L.pair_ptr, (const uint2*)L.rows, (uint2*)packed.p);
    APS_LAUNCHED();
  }
  // the only synchronisation before the end: the number of pairs and of correspondences size the RANSAC
  int64_t* h = (int64_t*)aps_ctx_stage(c, 16);
  if (!h) APS_FAIL(APS_ERR_ALLOC, "", "pinned staging allocation failed");
  APS_CUDA(cudaMemcpyAsync(h, sel.p + nsets, 16, cudaMemcpyDeviceToHost, s));
  APS_CUDA(cudaStreamSynchronize(s));
  const int64_t P = h[0], T = h[1];
  const size_t tot = (size_t)(T > 0 ? T : 1);
  APS_TRY(models.alloc((size_t)P * 9, s));
  APS_TRY(minv.alloc((size_t)P * 9, s));
  APS_TRY(inl.alloc(tot, s));
  APS_TRY(ni.alloc((size_t)P, s));
  APS_TRY(acc.alloc((size_t)P, s));
  APS_TRY(used.alloc((size_t)P, s));
  APS_TRY(am.alloc((size_t)P + 1, s));
  APS_TRY(am_rows.alloc(2 * tot, s));
  APS_TRY(ransac_chunks(c, P, T, pt.p, nullptr, packed.p, ii.p, jj.p, d_img_off, kp.p, keys.p, nullptr, 2 * (int64_t)max_trials,
                        seed, max_distance, confidence, max_trials, models.p, minv.p, inl.p, ni.p, acc.p, used.p));
  if (P > 0) {
    k_scan_counts<<<1, 1024, 0, s>>>(AcceptedInliers{acc.p, ni.p}, P, am.p, nullptr);
    APS_LAUNCHED();
    k_all_matches<<<(unsigned)P, 256, 0, s>>>(pt.p, (const uint2*)packed.p, inl.p, am.p, (uint2*)am_rows.p);
    APS_LAUNCHED();
  }
  // the download: [set_pair_ptr | pairs_lin | pt_ptr | match_ptr | (list pair_ptr) | models | models_inv | n_inliers |
  // draws_used | accepted] in pass order, then the allMatches rows (and the lists' rows)
  const size_t w64 = nt + (size_t)P + 2 * ((size_t)P + 1) + (want_lists ? (size_t)cells + 1 : 0) + 18 * (size_t)P;
  uint8_t* hs = (uint8_t*)aps_ctx_stage(c, w64 * 8 + (size_t)P * 9);
  if (!hs) APS_FAIL(APS_ERR_ALLOC, "", "pinned staging allocation failed");
  int64_t* h_spp = (int64_t*)hs;
  int64_t* h_lin = h_spp + nt;
  int64_t* h_pt = h_lin + P;
  int64_t* h_am = h_pt + P + 1;
  int64_t* h_pp = h_am + P + 1;
  double* h_models = (double*)(h_pp + (want_lists ? cells + 1 : 0));
  double* h_minv = h_models + 9 * P;
  int32_t* h_ni = (int32_t*)(h_minv + 9 * P);
  int32_t* h_used = h_ni + P;
  uint8_t* h_acc = (uint8_t*)(h_used + P);
  APS_CUDA(cudaMemcpyAsync(h_spp, sel.p, nt * 8, cudaMemcpyDeviceToHost, s));
  if (P > 0) {
    APS_CUDA(cudaMemcpyAsync(h_lin, lin.p, (size_t)P * 8, cudaMemcpyDeviceToHost, s));
    APS_CUDA(cudaMemcpyAsync(h_pt, pt.p, ((size_t)P + 1) * 8, cudaMemcpyDeviceToHost, s));
    APS_CUDA(cudaMemcpyAsync(h_am, am.p, ((size_t)P + 1) * 8, cudaMemcpyDeviceToHost, s));
    APS_CUDA(cudaMemcpyAsync(h_models, models.p, (size_t)P * 72, cudaMemcpyDeviceToHost, s));
    APS_CUDA(cudaMemcpyAsync(h_minv, minv.p, (size_t)P * 72, cudaMemcpyDeviceToHost, s));
    APS_CUDA(cudaMemcpyAsync(h_ni, ni.p, (size_t)P * 4, cudaMemcpyDeviceToHost, s));
    APS_CUDA(cudaMemcpyAsync(h_used, used.p, (size_t)P * 4, cudaMemcpyDeviceToHost, s));
    APS_CUDA(cudaMemcpyAsync(h_acc, acc.p, (size_t)P, cudaMemcpyDeviceToHost, s));
  } else {
    h_am[0] = 0;
  }
  if (want_lists) APS_CUDA(cudaMemcpyAsync(h_pp, L.pair_ptr, ((size_t)cells + 1) * 8, cudaMemcpyDeviceToHost, s));
  APS_CUDA(cudaStreamSynchronize(s));
  std::vector<uint32_t> h_am_rows((size_t)(2 * h_am[P]));
  std::vector<int64_t> pp;
  std::vector<uint32_t> rows_h;
  std::vector<double> met_h;
  if (want_lists) {
    pp.assign(h_pp, h_pp + cells + 1);
    rows_h.resize((size_t)(2 * pp[cells]));
    if (L.metric) met_h.resize((size_t)pp[cells]);
  }
  if (!h_am_rows.empty())
    APS_CUDA(cudaMemcpyAsync(h_am_rows.data(), am_rows.p, h_am_rows.size() * 4, cudaMemcpyDeviceToHost, s));
  if (!rows_h.empty()) APS_CUDA(cudaMemcpyAsync(rows_h.data(), L.rows, rows_h.size() * 4, cudaMemcpyDeviceToHost, s));
  if (!met_h.empty()) APS_CUDA(cudaMemcpyAsync(met_h.data(), L.metric, met_h.size() * 8, cudaMemcpyDeviceToHost, s));
  if (!h_am_rows.empty() || !rows_h.empty()) APS_CUDA(cudaStreamSynchronize(s));
  const std::vector<int64_t> spp(h_spp, h_spp + nt);
  reorder(order, spp, h_lin, h_pt, h_am, h_am_rows.data(), h_models, h_minv, h_ni, h_acc, h_used, r);
  if (want_lists) {
    r->lists.assign((size_t)nsets, nullptr);
    APS_TRY(sets_split_lists(nsets, pp, rows_h, L.metric ? &met_h : nullptr, L.cell_off, ns.data(), order.data(),
                             r->lists.data()));
  }
  return APS_OK;
}

int run_global(aps_ctx* c, int nsets, const int* set_images, const std::vector<int64_t>& img_first,
               const std::vector<int64_t>& set_rows, const void* const* desc, const int64_t* counts, int D, int dtype,
               int layout, int k, double ratio, int mutual, const KeypointSource& keypoints, int m, double max_distance,
               double confidence, int max_trials, uint64_t seed, int want_lists, bool dev, aps_image_matches* r) {
  cudaStream_t s = c->stream;
  int64_t F = 0;
  for (int64_t F_b : set_rows) F += F_b;
  GlobalLists L;
  if (F > 0) {
    APS_TRY(global_lists_device(c, nsets, set_images, img_first, set_rows, desc, counts, D, dtype, layout, k, ratio,
                                mutual, L, dev));
  } else {  // no descriptor anywhere: every putative count is 0 (partner selection still runs, imageMatching.m:75-100)
    for (int b = 0; b < nsets; ++b) L.order.push_back(b);
    L.cell_off.assign(1, 0);
    for (int b = 0; b < nsets; ++b) L.cell_off.push_back(L.cell_off.back() + (int64_t)set_images[b] * set_images[b]);
    const int64_t cells = L.cell_off.back();
    APS_TRY(L.counts_buf.alloc((size_t)cells + 1, s));
    APS_CUDA(cudaMemsetAsync(L.counts_buf.p, 0, ((size_t)cells + 1) * 8, s));
    L.pair_counts = L.pair_ptr = L.counts_buf.p;  // zero counts, zero offsets
  }
  // a query row yields at most one match row: F bounds the rows of the lists
  APS_TRY(match_lists(c, nsets, set_images, img_first, counts, F, keypoints, L, F, m, max_distance, confidence,
                      max_trials, seed, want_lists, r));
  if (F > 0) global_lists_stats(c, dtype, L);
  return APS_OK;
}

int run_pairwise(aps_ctx* c, int nsets, const int* set_images, const std::vector<int64_t>& img_first,
                 const void* const* desc, const int64_t* counts, int D, int dtype, int layout, double match_threshold,
                 double max_ratio, int method, int64_t subset, uint64_t subset_seed, const KeypointSource& keypoints,
                 int m, double max_distance, double confidence, int max_trials, uint64_t seed, int want_lists, bool dev,
                 aps_image_matches* r) {
  cudaStream_t s = c->stream;
  const int nimg = (int)img_first[nsets];
  int64_t F = 0;
  for (int g = 0; g < nimg; ++g) F += counts[g];
  GlobalLists L;
  for (int b = 0; b < nsets; ++b) L.order.push_back(b);  // the pass keeps the caller's set order
  int64_t M = 0;
  {
    PairwiseRows R;
    APS_TRY(pairwise_rows_device(c, nsets, set_images, desc, counts, nimg, D, dtype, layout, match_threshold,
                                 max_ratio, method, subset, subset_seed, R, dev));
    // the lists in cell order, as GlobalLists: counts scattered into zeroed cells, offsets scanned, rows placed
    L.cell_off = R.cell_off;
    const int64_t cells = L.cell_off.back(), np = R.npairs;
    M = R.M;
    DevBuf<int64_t> dtab;
    APS_TRY(L.counts_buf.alloc((size_t)cells + 1, s));
    APS_TRY(L.ptr_buf.alloc((size_t)cells + 1, s));
    APS_TRY(L.rows_buf.alloc((size_t)(M > 0 ? 2 * M : 2), s));
    if (want_lists) APS_TRY(L.metric_buf.alloc((size_t)(M > 0 ? M : 1), s));
    APS_CUDA(cudaMemsetAsync(L.counts_buf.p, 0, ((size_t)cells + 1) * 8, s));
    if (np > 0) {
      APS_TRY(dtab.alloc(R.tab.size(), s));
      APS_CUDA(cudaMemcpyAsync(dtab.p, R.tab.data(), R.tab.size() * 8, cudaMemcpyHostToDevice, s));
      k_scatter_counts<<<(unsigned)aps_ceil_div(np, 256), 256, 0, s>>>(dtab.p, np, L.counts_buf.p);
      APS_LAUNCHED();
    }
    k_scan_counts<<<1, 1024, 0, s>>>(CountOf{L.counts_buf.p}, cells, L.ptr_buf.p, nullptr);
    APS_LAUNCHED();
    if (np > 0) {
      k_place_rows<<<(unsigned)np, 128, 0, s>>>(dtab.p, np, L.ptr_buf.p, (const uint2*)R.rows.p, R.metric.p,
                                                (uint2*)L.rows_buf.p, want_lists ? L.metric_buf.p : nullptr);
      APS_LAUNCHED();
    }
  }  // the batch-ordered rows are released before the RANSAC allocates
  L.pair_counts = L.counts_buf.p;
  L.pair_ptr = L.ptr_buf.p;
  L.rows = L.rows_buf.p;
  L.metric = want_lists ? L.metric_buf.p : nullptr;
  // a query row can match once in every pair of its image: the pass's M rows bound the lists
  return match_lists(c, nsets, set_images, img_first, counts, F, keypoints, L, M, m, max_distance, confidence,
                     max_trials, seed, want_lists, r);
}

int keypoint_dtype(int kp_dtype) {
  if (kp_dtype != APS_KP_F64 && kp_dtype != APS_KP_F32)
    APS_FAIL(APS_ERR_TYPE, "", "kp_dtype must be APS_KP_F64 or APS_KP_F32 (got %d)", kp_dtype);
  return APS_OK;
}

// a result for nsets sets, filled by fill(r) when nsets > 0; *out set only on success
template <class Fill>
int new_result(int nsets, aps_image_matches** out, Fill fill) {
  aps_image_matches* r = new (std::nothrow) aps_image_matches();
  if (!r) APS_FAIL(APS_ERR_ALLOC, "", "out of host memory");
  r->nsets = nsets;
  r->set_pair_ptr.assign((size_t)nsets + 1, 0);
  r->pt_ptr.assign(1, 0);
  r->match_ptr.assign(1, 0);
  const int rc = nsets > 0 ? fill(r) : APS_OK;
  if (rc != APS_OK) {
    delete r;
    return rc;
  }
  *out = r;
  return APS_OK;
}

}  // namespace

extern "C" int aps_global_image_matching_sets(aps_ctx* c, int nsets, const int* set_images, const void* const* desc,
                                              const int64_t* counts, int D, int dtype, int layout, int k, double ratio,
                                              int use_bf, int mutual, const double* keypoints, int m,
                                              double max_distance, double confidence, int max_trials, uint64_t seed,
                                              int want_lists, aps_image_matches** out) {
  (void)use_bf;
  // arguments first (the ids of aps_feature_matching_global_sets, then the RANSAC parameters), then the device
  if (!out) APS_FAIL(APS_ERR_ARGS, "", "out is NULL");
  *out = nullptr;
  std::vector<int64_t> img_first, set_rows;
  APS_TRY(global_sets_args(nsets, set_images, counts, D, dtype, k, img_first, set_rows));
  APS_TRY(ransac_params(2 * (int64_t)max_trials, max_trials, confidence));
  int64_t F = 0;
  for (int64_t F_b : set_rows) F += F_b;
  if (F > 0 && !keypoints) APS_FAIL(APS_ERR_ARGS, "", "keypoints is NULL");
  APS_CTX(c);
  return new_result(nsets, out, [&](aps_image_matches* r) {
    return run_global(c, nsets, set_images, img_first, set_rows, desc, counts, D, dtype, layout, k, ratio, mutual,
                      {keypoints, false, APS_KP_F64}, m, max_distance, confidence, max_trials, seed, want_lists, false,
                      r);
  });
}

extern "C" int aps_global_image_matching_sets_dev(aps_ctx* c, int nsets, const int* set_images, const void* d_pooled,
                                                  const int64_t* counts, int D, int dtype, int k, double ratio,
                                                  int use_bf, int mutual, const void* d_keypoints, int kp_dtype, int m,
                                                  double max_distance, double confidence, int max_trials,
                                                  uint64_t seed, int want_lists, void* producer_stream,
                                                  aps_image_matches** out) {
  (void)use_bf;
  // the host entry's arguments, then the keypoint type, the device pointers, the context and the hand-off
  if (!out) APS_FAIL(APS_ERR_ARGS, "", "out is NULL");
  *out = nullptr;
  std::vector<int64_t> img_first, set_rows;
  APS_TRY(global_sets_args(nsets, set_images, counts, D, dtype, k, img_first, set_rows));
  APS_TRY(ransac_params(2 * (int64_t)max_trials, max_trials, confidence));
  int64_t F = 0;
  for (int64_t F_b : set_rows) F += F_b;
  if (F > 0 && !d_keypoints) APS_FAIL(APS_ERR_ARGS, "", "keypoints is NULL");
  APS_TRY(keypoint_dtype(kp_dtype));
  APS_TRY(dev_inputs(c, F, d_pooled, d_keypoints, producer_stream));
  const std::vector<const void*> ptrs =
      pooled_image_ptrs(d_pooled, counts, img_first[nsets], D, dtype == APS_F32 ? 4 : 1);
  return new_result(nsets, out, [&](aps_image_matches* r) {
    return run_global(c, nsets, set_images, img_first, set_rows, ptrs.data(), counts, D, dtype, APS_ROW_MAJOR, k, ratio,
                      mutual, {d_keypoints, true, kp_dtype}, m, max_distance, confidence, max_trials, seed,
                      want_lists, true, r);
  });
}

extern "C" int aps_global_image_matching(aps_ctx* c, const void* const* desc, const int64_t* counts, int n, int D,
                                         int dtype, int layout, int k, double ratio, int use_bf, int mutual,
                                         const double* keypoints, int m, double max_distance, double confidence,
                                         int max_trials, uint64_t seed, int want_lists, aps_image_matches** out) {
  return aps_global_image_matching_sets(c, 1, &n, desc, counts, D, dtype, layout, k, ratio, use_bf, mutual, keypoints,
                                        m, max_distance, confidence, max_trials, seed, want_lists, out);
}

extern "C" int aps_pairwise_image_matching_sets(aps_ctx* c, int nsets, const int* set_images, const void* const* desc,
                                                const int64_t* counts, int D, int dtype, int layout,
                                                double match_threshold, double max_ratio, int method, int64_t subset,
                                                uint64_t subset_seed, const double* keypoints, int m,
                                                double max_distance, double confidence, int max_trials, uint64_t seed,
                                                int want_lists, aps_image_matches** out) {
  // arguments first (the statuses of aps_feature_matching_pairwise_sets, then the RANSAC parameters), then the device
  std::vector<int64_t> img_first;
  APS_TRY(pairwise_sets_args(nsets, set_images, counts, D, dtype, method, subset, img_first));
  APS_TRY(ransac_params(2 * (int64_t)max_trials, max_trials, confidence));
  int64_t F = 0;
  for (int64_t g = 0; g < img_first[nsets]; ++g) F += counts[g];
  if (F > 0 && !keypoints) APS_FAIL(APS_ERR_ARGS, "", "keypoints is NULL");
  if (!out) APS_FAIL(APS_ERR_ARGS, "", "out is NULL");
  *out = nullptr;
  APS_CTX(c);
  return new_result(nsets, out, [&](aps_image_matches* r) {
    return run_pairwise(c, nsets, set_images, img_first, desc, counts, D, dtype, layout, match_threshold, max_ratio,
                        method, subset, subset_seed, {keypoints, false, APS_KP_F64}, m, max_distance, confidence,
                        max_trials, seed, want_lists, false, r);
  });
}

extern "C" int aps_pairwise_image_matching_sets_dev(aps_ctx* c, int nsets, const int* set_images, const void* d_pooled,
                                                    const int64_t* counts, int D, int dtype, double match_threshold,
                                                    double max_ratio, int method, int64_t subset, uint64_t subset_seed,
                                                    const void* d_keypoints, int kp_dtype, int m, double max_distance,
                                                    double confidence, int max_trials, uint64_t seed, int want_lists,
                                                    void* producer_stream, aps_image_matches** out) {
  // the host entry's arguments, then the keypoint type, the device pointers, the context and the hand-off
  std::vector<int64_t> img_first;
  APS_TRY(pairwise_sets_args(nsets, set_images, counts, D, dtype, method, subset, img_first));
  APS_TRY(ransac_params(2 * (int64_t)max_trials, max_trials, confidence));
  int64_t F = 0;
  for (int64_t g = 0; g < img_first[nsets]; ++g) F += counts[g];
  if (F > 0 && !d_keypoints) APS_FAIL(APS_ERR_ARGS, "", "keypoints is NULL");
  if (!out) APS_FAIL(APS_ERR_ARGS, "", "out is NULL");
  *out = nullptr;
  APS_TRY(keypoint_dtype(kp_dtype));
  APS_TRY(dev_inputs(c, F, d_pooled, d_keypoints, producer_stream));
  const std::vector<const void*> ptrs =
      pooled_image_ptrs(d_pooled, counts, img_first[nsets], D, dtype == APS_F32 ? 4 : 1);
  return new_result(nsets, out, [&](aps_image_matches* r) {
    return run_pairwise(c, nsets, set_images, img_first, ptrs.data(), counts, D, dtype, APS_ROW_MAJOR, match_threshold,
                        max_ratio, method, subset, subset_seed, {d_keypoints, true, kp_dtype}, m, max_distance,
                        confidence, max_trials, seed, want_lists, true, r);
  });
}

extern "C" int aps_pairwise_image_matching(aps_ctx* c, const void* const* desc, const int64_t* counts, int n, int D,
                                           int dtype, int layout, double match_threshold, double max_ratio, int method,
                                           int64_t subset, uint64_t subset_seed, const double* keypoints, int m,
                                           double max_distance, double confidence, int max_trials, uint64_t seed,
                                           int want_lists, aps_image_matches** out) {
  return aps_pairwise_image_matching_sets(c, 1, &n, desc, counts, D, dtype, layout, match_threshold, max_ratio, method,
                                          subset, subset_seed, keypoints, m, max_distance, confidence, max_trials,
                                          seed, want_lists, out);
}

extern "C" int aps_image_matches_nsets(const aps_image_matches* r) { return r ? r->nsets : 0; }
extern "C" int64_t aps_image_matches_pairs(const aps_image_matches* r) {
  return r ? (int64_t)r->pairs_lin.size() : 0;
}
extern "C" const int64_t* aps_image_matches_set_pair_ptr(const aps_image_matches* r) {
  return r ? r->set_pair_ptr.data() : nullptr;
}
extern "C" const int64_t* aps_image_matches_pairs_lin(const aps_image_matches* r) {
  return r ? r->pairs_lin.data() : nullptr;
}
extern "C" const int64_t* aps_image_matches_pt_ptr(const aps_image_matches* r) { return r ? r->pt_ptr.data() : nullptr; }
extern "C" const int64_t* aps_image_matches_match_ptr(const aps_image_matches* r) {
  return r ? r->match_ptr.data() : nullptr;
}
extern "C" const uint32_t* aps_image_matches_match_rows(const aps_image_matches* r) {
  return r ? r->match_rows.data() : nullptr;
}
extern "C" const double* aps_image_matches_models(const aps_image_matches* r) { return r ? r->models.data() : nullptr; }
extern "C" const double* aps_image_matches_models_inv(const aps_image_matches* r) {
  return r ? r->models_inv.data() : nullptr;
}
extern "C" const int32_t* aps_image_matches_n_inliers(const aps_image_matches* r) {
  return r ? r->n_inliers.data() : nullptr;
}
extern "C" const uint8_t* aps_image_matches_accepted(const aps_image_matches* r) {
  return r ? r->accepted.data() : nullptr;
}
extern "C" const int32_t* aps_image_matches_draws_used(const aps_image_matches* r) {
  return r ? r->draws_used.data() : nullptr;
}
extern "C" const aps_matchlist* aps_image_matches_list(const aps_image_matches* r, int b) {
  return r && b >= 0 && b < (int)r->lists.size() ? r->lists[b] : nullptr;
}
extern "C" void aps_image_matches_free(aps_image_matches* r) { delete r; }
