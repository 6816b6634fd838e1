// aps_rerank.cu -- K3: exact FP32 re-rank of the tensor-core candidates + completeness proof.
//
// The tcgen05 pass (aps_knn_tc.cu) ranks train rows by an APPROXIMATE score (bf16 operands).  The
// reference contract (PP/mex/flann_knn.cpp:229-252, matchFeaturesScratch.m:351-362) is the exact
// ordering, so every candidate's distance is recomputed here with the oracle's own operation order
// and the row's top-k is PROVEN complete:
//
//   approx distance  s~(score) = alpha_row + beta_row * score        (monotone decreasing in score)
//   |s~ - s_exact| <= eps  for every train row (bound derived in DESIGN.md "Exactness")
//   every row that is not a candidate has s~ >= W := min over segments of the worst retained s~
//   => if  W - eps > (k-th smallest exact candidate distance)  no outsider can enter or tie the top-k.
//
// Rows failing the test are appended to a list and re-searched by the exact CUDA-core kernel.
// Tile mode (lists made by the segment epilogue of the per-pair searches): W per list = its third entry, and the one
// segment whose two best both sit in a list is scanned exactly by the row's lanes (see the W computation below).
// One warp per query row, one lane per candidate (nseg*kcand <= 32), or two per lane for up to 64 candidates (the K' = 16
// lists of 6 <= k <= 12; no tile mode, no pairwise shortcut).
#include <math_constants.h>

#include "aps_common.cuh"
#include "aps_exact_math.cuh"

namespace {

// G lanes per query row (G = 8, 16 or 32; G * C >= number of candidates): 32/G rows per warp.  C candidates per lane:
// candidate e sits in lane e % G, register e / G.
template <int G, int C = 1>
__global__ void __launch_bounds__(256) k_rerank(const float* __restrict__ Q, const float* __restrict__ sqQ,
                                                const float* __restrict__ invnQ, const float* __restrict__ T,
                                                const float* __restrict__ sqT, int D, int metric, int64_t q0,
                                                int64_t nq, int64_t t0, int nseg, int kcand,
                                                const uint32_t* __restrict__ cand_idx,
                                                const float* __restrict__ cand_score,
                                                const int32_t* __restrict__ flags, int bias_mode, int k,
                                                int64_t out_row0, uint32_t* __restrict__ idx,
                                                float* __restrict__ dist, int32_t* __restrict__ fb_rows,
                                                int32_t* __restrict__ fb_count, aps_pair_tables pt,
                                                const int32_t* __restrict__ row_map,
                                                const int32_t* __restrict__ nrows_dev,
                                                const int32_t* __restrict__ perm, int cand_stride,
                                                int kcap_exact) {
  constexpr int RPW = 32 / G;  // rows per warp
  if (nrows_dev && (int64_t)blockIdx.x * (blockDim.x >> 5) * RPW >= (int64_t)(*nrows_dev)) return;  // second pass: short list
  const int lane = threadIdx.x & 31, sub = lane / G, sl = lane % G;
  const unsigned segmask = (G == 32) ? 0xffffffffu : (((1u << G) - 1u) << (sub * G));
  const int64_t r = ((int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * RPW + sub;
  const bool row_ok = r < (nrows_dev ? (int64_t)(*nrows_dev) : nq);
  int64_t q = q0 + (row_ok ? r : 0);
  if (row_map) q = row_ok ? (int64_t)row_map[r] : q0;  // second pass: candidate row r belongs to query row_map[r]
  int64_t orow = q - out_row0;  // output row
  int64_t tn = 0;               // batched pairwise: rows of the train image
  if (pt.eoff) {  // batched pairwise: candidate row r is entry r of pair p: query off_i + (r - eoff[p]), train image j
    const int64_t e = row_ok ? r : 0;
    int lo = 0, hi = pt.npairs;  // last p with eoff[p] <= e
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (pt.eoff[mid] <= e) lo = mid; else hi = mid;
    }
    q = (int64_t)pt.qoff[lo] + (e - pt.eoff[lo]);
    t0 = pt.toff[lo];
    tn = pt.tcnt[lo];
    orow = e;
  }
  const int ncand = nseg * kcand;
  // tile mode: keys carry the column in their 7 low mantissa bits: |key - score| <= 2^-16 |score| <= 1.5e-5 * (|a.b| + |bias|)
  // <= 2.3e-5 * max|x|^2, times |beta| = 2
  const float eps = eps_bound(flags, bias_mode, pt.operand_fp16) +
                    (pt.tile_mode ? 5.0e-5f * fmaxf(__int_as_float(flags[2]), 1.0f) : 0.0f);
  const bool exact = flags[0] != 0 && pt.operand_fp16 != 1;  // (bf16 path) operand = raw row, per-row scale: beta carries 1/norm; pairwise: invn = 1
  const float a2 = sqQ[q];
  // s~ = alpha + beta*score
  const float alpha = bias_mode ? a2 : __fadd_rn(a2, 1.0f);
  const float beta = bias_mode ? -2.0f : (exact ? -2.0f * invnQ[q] : -2.0f);

  uint32_t ci[C];
  bool valid[C];
  float sapx[C];
#pragma unroll
  for (int j = 0; j < C; ++j) {
    const int e = j * G + sl;
    ci[j] = 0xffffffffu;
    float sc = -CUDART_INF_F;
    if (row_ok && e < ncand) {
      ci[j] = cand_idx[r * cand_stride + e];  // cand_stride > ncand: only the row's first nseg lists are read
      sc = cand_score[r * cand_stride + e];
      if (perm && ci[j] != 0xffffffffu) ci[j] = (uint32_t)perm[ci[j]];  // position in the sorted train view -> original row
    }
    valid[j] = ci[j] != 0xffffffffu;
    sapx[j] = valid[j] ? fmaf(beta, sc, alpha) : CUDART_INF_F;  // monotone in sc; its own rounding is inside eps
  }

  // W = min over lists of the worst (largest) retained approx distance
  float W = CUDART_INF_F;
  uint32_t segscan[2] = {0xffffffffu, 0xffffffffu}, segskip[4] = {0u, 0u, 0u, 0u};  // tile mode: segments to scan exactly
  if (C == 1 && pt.tile_mode) {
    // lists of three sorted by approximate score (best first), each the top-3 of "two best per segment": a column
    // outside list s is bounded by the list's third entry, or by its second when the two best share a segment;
    // a list that is not full bounds its outsiders by its last entry (conservative: tiny train images only)
    for (int s = 0; s < nseg; ++s) {
      const uint32_t c0 = __shfl_sync(0xffffffffu, ci[0], s * 3, G), c1 = __shfl_sync(0xffffffffu, ci[0], s * 3 + 1, G);
      const uint32_t c2 = __shfl_sync(0xffffffffu, ci[0], s * 3 + 2, G);
      const float a0 = __shfl_sync(0xffffffffu, sapx[0], s * 3, G), a1 = __shfl_sync(0xffffffffu, sapx[0], s * 3 + 1, G);
      const float a2 = __shfl_sync(0xffffffffu, sapx[0], s * 3 + 2, G);
      float w;
      if (c0 == 0xffffffffu) w = CUDART_INF_F;        // no selectable column in this list's part of the train range
      else if (c1 == 0xffffffffu) w = a0;
      else if (c2 == 0xffffffffu) w = a1;
      else {
        w = a2;
        // two best from one segment: the segment's other columns are only bounded by a1.  Instead of giving up, the
        // row's lanes scan that one segment exactly further down (segscan) -- 64 columns, not the whole image.
        if (c0 / (uint32_t)pt.tile_mode == c1 / (uint32_t)pt.tile_mode) {
          if (segscan[0] == 0xffffffffu) { segscan[0] = c0 / (uint32_t)pt.tile_mode; segskip[0] = c0; segskip[1] = c1; }
          else if (segscan[1] == 0xffffffffu) { segscan[1] = c0 / (uint32_t)pt.tile_mode; segskip[2] = c0; segskip[3] = c1; }
          else w = a1;
        }
      }
      W = fminf(W, w);
    }
  } else {
    // entries a list can hold: the tensor pass keeps only kcap_exact of the kcand slots when the operands are exact
    // (aps_knn_tc.cu, variant chosen by the same device flag).  Slots beyond that capacity say nothing; an EMPTY slot
    // inside the capacity means every column of the list's range is a candidate (W = +inf).
    const int cap = (kcap_exact > 0 && flags[0] != 0) ? kcap_exact : kcand;
    for (int s = 0; s < nseg; ++s) {
      float m = (sl >= s * kcand && sl < s * kcand + cap) ? sapx[0] : -CUDART_INF_F;
#pragma unroll
      for (int j = 1; j < C; ++j) {
        const int e = j * G + sl;
        m = fmaxf(m, (e >= s * kcand && e < s * kcand + cap) ? sapx[j] : -CUDART_INF_F);
      }
#pragma unroll
      for (int o = G / 2; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o, G));
      W = fminf(W, m);
    }
  }
  // prune: lanes whose lower bound exceeds the k-th smallest upper bound cannot be in the top-k
  float ub[C], lb[C];
  int below[C];
#pragma unroll
  for (int j = 0; j < C; ++j) {
    ub[j] = sapx[j] + eps;
    lb[j] = sapx[j] - eps;
    below[j] = 0;
  }
  for (int l = 0; l < G; ++l) {
#pragma unroll
    for (int jj = 0; jj < C; ++jj) {
      float o = __shfl_sync(0xffffffffu, ub[jj], l, G);
#pragma unroll
      for (int j = 0; j < C; ++j) below[j] += (o < lb[j]);
    }
  }
  // batched pairwise shortcut: rejection of the row by the ratio / threshold test proven from the approximate
  // distances alone: exact d1 >= m1 - eps (rows outside the list have s~ >= W >= m1) and exact d2 <= m2 + eps
  bool rej = false;
  if (C == 1 && pt.prune) {
    float m1 = sapx[0];
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) m1 = fminf(m1, __shfl_xor_sync(0xffffffffu, m1, o, G));
    const unsigned eq = __ballot_sync(0xffffffffu, sapx[0] == m1) & segmask;
    float m2 = (eq != 0u && lane == __ffs(eq) - 1) ? CUDART_INF_F : sapx[0];  // drop ONE instance of the minimum
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) m2 = fminf(m2, __shfl_xor_sync(0xffffffffu, m2, o, G));
    if (m2 < CUDART_INF_F) {  // at least two candidates
      const double lb1 = (double)m1 - (double)eps, ub2 = (double)m2 + (double)eps;
      const double slack = 1e-6 * (fabs(lb1) + 1.0);
      rej = (lb1 > pt.prune_r2 * ub2 + slack) || (lb1 > pt.prune_mt + slack);
    }
  }
  bool need[C], nan_mine = false;
  float d[C];   // ranking key
  float ds[C];  // the same distance in the domain of the approximate scores (squared), for the proof
#pragma unroll
  for (int j = 0; j < C; ++j) {
    need[j] = valid[j] && below[j] < k && !rej;
    d[j] = CUDART_INF_F;
    ds[j] = CUDART_INF_F;
    if (need[j]) {
      const float* a = Q + q * D;
      const float* b = T + (int64_t)ci[j] * D;
      if (metric == 2) {      // Euclidean search ('kdtree' / 'subsetpdist2'): rank by r = sqrt(s), ties -> lower index
        ds[j] = l2sq_seq(a, b, D);
        d[j] = __fsqrt_rn(ds[j]);
      } else if (metric == 3) {   // 'pca2nn': [sim1, id1] = max(G, [], 2): rank by similarity (descending), first index on ties
        const float sim = dot_seq(a, b, D);
        d[j] = -sim;
        ds[j] = __fsub_rn(2.0f, __fmul_rn(2.0f, sim));   // d1Block = single(2 - 2*sim1), :568-570
      } else {
        d[j] = (metric == 0) ? l2sq_flann(a, b, D) : ssd_seq(a, b, D, a2, sqT[ci[j]]);
        ds[j] = d[j];
      }
    }
    nan_mine = nan_mine || (need[j] && !(d[j] == d[j]));
  }
  const bool nan_seen = (__ballot_sync(0xffffffffu, nan_mine) & segmask) != 0u;
  // rank by (distance, index)
  int rank[C];
#pragma unroll
  for (int j = 0; j < C; ++j) rank[j] = 0;
  for (int l = 0; l < G; ++l) {
#pragma unroll
    for (int jj = 0; jj < C; ++jj) {
      float od = __shfl_sync(0xffffffffu, d[jj], l, G);
      uint32_t oi = __shfl_sync(0xffffffffu, ci[jj], l, G);
      bool oneed = __shfl_sync(0xffffffffu, (int)need[jj], l, G);
#pragma unroll
      for (int j = 0; j < C; ++j) rank[j] += oneed && (od < d[j] || (od == d[j] && oi < ci[j]));
    }
  }
  int nvalid = 0;
#pragma unroll
  for (int j = 0; j < C; ++j) nvalid += __popc(__ballot_sync(0xffffffffu, need[j]) & segmask);
#pragma unroll
  for (int j = 0; j < C; ++j) {
    if (need[j] && rank[j] < k) {
      idx[orow * k + rank[j]] = (uint32_t)((int64_t)ci[j] - t0 + 1);
      dist[orow * k + rank[j]] = (metric == 2) ? __fmul_rn(d[j], d[j]) : (metric == 3 ? ds[j] : d[j]);   // :146-147, :153-154: dBest = d.^2
    }
  }
#pragma unroll
  for (int j = 0; j < C; ++j) {
    const int e = j * G + sl;
    if (row_ok && e >= nvalid && e < k) {  // fewer than k neighbours exist: flann_knn.cpp:216-219
      idx[orow * k + e] = 0u;
      dist[orow * k + e] = CUDART_INF_F;
    }
  }
  // completeness proof
  float dk = -CUDART_INF_F;  // k-th smallest exact distance (or -inf when fewer than k candidates)
  {
    float mine = (need[0] && rank[0] == k - 1) ? ds[0] : -CUDART_INF_F;
#pragma unroll
    for (int j = 1; j < C; ++j) mine = fmaxf(mine, (need[j] && rank[j] == k - 1) ? ds[j] : -CUDART_INF_F);
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) mine = fmaxf(mine, __shfl_xor_sync(0xffffffffu, mine, o, G));
    dk = mine;
    // metric 2 ranks by sqrt_rn(s): an outsider must exceed s_k by more than what two roundings can merge
    if (metric == 2 && dk > 0.f) dk = dk * (1.0f + 1.0e-6f);
  }
  bool proven;
  if (nvalid >= k)
    proven = (W - eps > dk);
  else
    proven = (W == CUDART_INF_F);  // every train row was a candidate
  if (C == 1 && pt.tile_mode) {
    // segments whose two best both sit in a list: every other column of the segment must be farther than the k-th
    // neighbour, checked with exact distances (strictly: a tie would have to be ranked by index)
    const bool want = row_ok && proven && !rej && segscan[0] != 0xffffffffu;
    if (__any_sync(0xffffffffu, want)) {
      float dmin = CUDART_INF_F;
      bool bad = false;
      if (want) {
        if (nvalid < k || !pt.eoff) bad = true;
        for (int z = 0; z < 2 && !bad; ++z) {
          if (segscan[z] == 0xffffffffu) break;
          const int64_t cbeg = (int64_t)segscan[z] * pt.tile_mode;
          const int64_t c_lo = cbeg > t0 ? cbeg : t0, c_hi = (cbeg + pt.tile_mode < t0 + tn) ? cbeg + pt.tile_mode : t0 + tn;
          const float* a = Q + q * D;
          for (int64_t col = c_lo + sl; col < c_hi; col += G) {
            if ((uint32_t)col == segskip[2 * z] || (uint32_t)col == segskip[2 * z + 1]) continue;
            const float* b = T + col * D;
            const float dd = (metric == 0)   ? l2sq_flann(a, b, D)
                             : (metric == 2) ? l2sq_seq(a, b, D)
                             : (metric == 3) ? __fsub_rn(2.0f, __fmul_rn(2.0f, dot_seq(a, b, D)))
                                             : ssd_seq(a, b, D, a2, sqT[col]);
            if (!(dd == dd)) bad = true;
            dmin = fminf(dmin, dd);
          }
        }
      }
#pragma unroll
      for (int o = G / 2; o > 0; o >>= 1) dmin = fminf(dmin, __shfl_xor_sync(0xffffffffu, dmin, o, G));
      const bool anybad = (__ballot_sync(0xffffffffu, bad) & segmask) != 0u;
      if (want && (anybad || !(dmin > dk))) proven = false;
    }
  }
  if (rej) proven = true;  // nothing to prove: the row is reported as having no neighbour
  if (nan_seen) proven = false;
  if (row_ok && !proven && sl == 0) {
    int pos = atomicAdd(fb_count, 1);
    fb_rows[pos] = (int32_t)(pt.eoff ? orow : q);
  }
}

}  // namespace

int aps_k_rerank(cudaStream_t s, const float* Q, const float* sqQ, const float* invnQ, const float* T,
                 const float* sqT, int D, int metric, int64_t q0, int64_t nq, int64_t t0, int nseg, int kcand,
                 const uint32_t* cand_idx, const float* cand_score, const int32_t* exact_flag, int bias_mode,
                 const int32_t* flags, int k, int64_t out_row0, uint32_t* idx, float* dist, int32_t* fb_rows,
                 int32_t* fb_count, const aps_pair_tables* pairs, const int32_t* row_map, const int32_t* nrows_dev,
                 const int32_t* perm, int cand_stride, int kcap_exact) {
  (void)exact_flag;
  if (nq == 0) return APS_OK;
  aps_pair_tables pt;
  memset(&pt, 0, sizeof pt);
  if (pairs) pt = *pairs;
  const int ncand = nseg * kcand;
  if (ncand > 64 || (ncand > 32 && (pt.tile_mode || pt.prune))) {
    aps_set_error(APS_ERR_ARGS, "", "rerank: nseg*kcand must be <= 64 (<= 32 in tile mode or with the pairwise shortcut)");
    return APS_ERR_ARGS;
  }
  if (cand_stride <= 0) cand_stride = ncand;
  if (k > 16 || k > ncand) {
    aps_set_error(APS_ERR_ARGS, "", "rerank: k must be <= min(16, candidates)");
    return APS_ERR_ARGS;
  }
#define APS_RERANK(G, C)                                                                                           \
  k_rerank<G, C><<<(unsigned)aps_ceil_div(nq, 8 * (32 / G)), 256, 0, s>>>(Q, sqQ, invnQ, T, sqT, D, metric, q0, nq, t0, \
                                                                       nseg, kcand, cand_idx, cand_score, flags,     \
                                                                       bias_mode, k, out_row0, idx, dist, fb_rows,  \
                                                                       fb_count, pt, row_map, nrows_dev, perm,       \
                                                                       cand_stride, kcap_exact)
  if (ncand <= 8) APS_RERANK(8, 1);
  else if (ncand <= 16) APS_RERANK(16, 1);
  else if (ncand <= 32) APS_RERANK(32, 1);
  else APS_RERANK(32, 2);
#undef APS_RERANK
  APS_LAUNCHED();
  return APS_OK;
}
