// aps_filter.cu -- K5: per-feature filters and deterministic compaction into the match-list cell
// order; K6: top-m image-partner selection.
//
// Replaces  the interpreted loop PP/featureMatching/featureMatchingGlobal.m:123-161 (self / same-image
//           removal, ratio test, append to matches{min,max}), the filters and greedy uniqueness of
//           PP/featureMatching/matchFeaturesScratch.m:169-211, and PP/imageMatching/imageMatching.m:75-100.
//
// HBM-streaming integer work: the filter reads k*(4+4) bytes per query and writes 8; compaction
// reads/writes 8-16 bytes per query.  Output order is defined by the reference's loop order, so the
// compaction is a stable counting sort keyed by (cell, query order), not an atomic append.
#include <math_constants.h>

#include "aps_common.cuh"

// ------------------------------------------------------------------------------------------------
// K5a  featureMatchingGlobal.m:123-147.  idx/dist row-major [.. x k], rows indexed from q0.
__global__ void k_global_filter(const uint32_t* __restrict__ idx, const float* __restrict__ dist, int k, int64_t q0,
                                int64_t q1, const int32_t* __restrict__ img_of_row,
                                const int64_t* __restrict__ img_off, float ratio_thr, int2* __restrict__ records) {
  int64_t q = q0 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= q1) return;
  const int32_t qi = img_of_row[q];
  float sd0 = 0.f, sd1 = 0.f;
  uint32_t s0 = 0;
  int ns = 0;
  for (int c = 0; c < k && ns < 2; ++c) {
    uint32_t j = idx[q * k + c];
    if (j == 0u) continue;                    // missing neighbour (k > F)
    if (j == (uint32_t)(q + 1)) continue;     // :130 self, by INDEX
    if (img_of_row[j - 1] == qi) continue;    // :135 same image
    float d = dist[q * k + c];
    if (ns == 0) {
      sd0 = d;
      s0 = j;
    } else {
      sd1 = d;
    }
    ++ns;
  }
  int32_t t = 0;
  uint32_t p = 0;
  if (ns == 2) {
    // :145  single / single, compared with the threshold in single precision (MATLAB converts the
    // double operand of a mixed comparison to single)
    float ratio = __fdiv_rn(sd0, fmaxf(sd1, APS_EPS32));
    if (!(ratio > ratio_thr)) {
      int32_t ti = img_of_row[s0 - 1];
      t = ti + 1;
      p = (uint32_t)((int64_t)(s0 - 1) - img_off[ti] + 1);
    }
  }
  records[q] = make_int2(t, (int32_t)p);  // one 8-byte record per query: (target image + 1 | 0, partner's local index)
}

int aps_k_global_filter(cudaStream_t s, const uint32_t* idx, const float* dist, int k, int64_t q0, int64_t q1,
                        const int32_t* img_of_row, const int64_t* img_off, float ratio_thr, int2* records) {
  if (q1 <= q0) return APS_OK;
  k_global_filter<<<(unsigned)aps_ceil_div(q1 - q0, 256), 256, 0, s>>>(idx, dist, k, q0, q1, img_of_row, img_off,
                                                                      ratio_thr, records);
  APS_LAUNCHED();
  return APS_OK;
}

// opt-in cross-check of the records: two passes so that every decision reads the ORIGINAL records
__global__ void k_records_mutual_mark(const int2* __restrict__ rec, const int32_t* __restrict__ img_of_row,
                                      const int64_t* __restrict__ img_off, int64_t F, uint8_t* __restrict__ keep) {
  const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= F) return;
  const int2 r = rec[q];
  uint8_t k = 0;
  if (r.x > 0) {
    const int64_t g = img_off[r.x - 1] + (int64_t)(uint32_t)r.y - 1;   // global row of the matched feature
    const int2 b = rec[g];
    k = (b.x == img_of_row[q] + 1) && ((int64_t)(uint32_t)b.y == q - img_off[img_of_row[q]] + 1);
  }
  keep[q] = k;
}
__global__ void k_records_mutual_apply(int2* __restrict__ rec, int64_t F, const uint8_t* __restrict__ keep) {
  const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (q < F && !keep[q]) rec[q] = make_int2(0, 0);
}
int aps_k_records_mutual(cudaStream_t s, int2* records, const int32_t* img_of_row, const int64_t* img_off, int64_t F,
                         uint8_t* keep) {
  if (F == 0) return APS_OK;
  const unsigned grid = (unsigned)aps_ceil_div(F, 256);
  k_records_mutual_mark<<<grid, 256, 0, s>>>(records, img_of_row, img_off, F, keep);
  APS_LAUNCHED();
  k_records_mutual_apply<<<grid, 256, 0, s>>>(records, F, keep);
  APS_LAUNCHED();
  return APS_OK;
}

// ------------------------------------------------------------------------------------------------
// K5b  compaction.  Cell (a,b), a<b, holds first the accepted queries of image a (ascending local
// index) then those of image b -- i.e. ascending GLOBAL query order.  One warp walks one image's
// queries in order and hands out, per target image, consecutive ranks (warp match + popc).
__global__ void k_rank_per_image(const int2* __restrict__ records, const int64_t* __restrict__ img_off, int n,
                                 int64_t* __restrict__ dir_counts, int64_t* __restrict__ rank) {
  extern __shared__ int cnt[];  // [n]
  const int i = blockIdx.x, lane = threadIdx.x;
  for (int t = lane; t < n; t += 32) cnt[t] = 0;
  __syncwarp();
  const int64_t b = img_off[i], e = img_off[i + 1];
  for (int64_t base = b; base < e; base += 32) {
    const int64_t q = base + lane;
    const int t = (q < e) ? records[q].x : 0;
    const bool active = t > 0;
    const unsigned amask = __ballot_sync(0xffffffffu, active);
    int myrank = 0, cbase = 0;
    unsigned peers = 0;
    if (active) {
      peers = __match_any_sync(amask, t);
      cbase = cnt[t - 1];
      myrank = __popc(peers & ((1u << lane) - 1u));
    }
    __syncwarp();
    if (active) {
      rank[q] = (int64_t)cbase + myrank;
      if (myrank == 0) cnt[t - 1] = cbase + __popc(peers);
    }
    __syncwarp();
  }
  for (int t = lane; t < n; t += 32) dir_counts[(int64_t)i * n + t] = cnt[t];
}

// Same result with 8 warps per image (n <= 1024 targets): pass 1 counts per (warp sub-range, target), a
// prefix over the sub-ranges gives every warp its starting rank, pass 2 hands the ranks out.
constexpr int RPI_WARPS = 8;
__global__ void __launch_bounds__(32 * RPI_WARPS) k_rank_per_image_mw(const int2* __restrict__ records,
                                                                       const int64_t* __restrict__ img_off, int n,
                                                                       int64_t* __restrict__ dir_counts,
                                                                       int64_t* __restrict__ rank) {
  extern __shared__ int cnt[];  // [RPI_WARPS][n]
  const int i = blockIdx.x, lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int t = threadIdx.x; t < RPI_WARPS * n; t += blockDim.x) cnt[t] = 0;
  __syncthreads();
  const int64_t b = img_off[i], e = img_off[i + 1];
  const int64_t per = (((e - b) + RPI_WARPS - 1) / RPI_WARPS + 31) / 32 * 32;
  const int64_t wb = min(e, b + w * per), we = min(e, wb + per);
  int* mine = cnt + w * n;
  for (int pass = 0; pass < 2; ++pass) {
    for (int64_t base = wb; base < we; base += 32) {
      const int64_t q = base + lane;
      const int t = (q < we) ? records[q].x : 0;
      const bool active = t > 0;
      const unsigned amask = __ballot_sync(0xffffffffu, active);
      int myrank = 0, cbase = 0;
      unsigned peers = 0;
      if (active) {
        peers = __match_any_sync(amask, t);
        cbase = mine[t - 1];
        myrank = __popc(peers & ((1u << lane) - 1u));
      }
      __syncwarp();
      if (active) {
        if (pass == 1) rank[q] = (int64_t)cbase + myrank;
        if (myrank == 0) mine[t - 1] = cbase + __popc(peers);
      }
      __syncwarp();
    }
    __syncthreads();
    if (pass == 0) {  // counts -> exclusive prefix over the warp sub-ranges; totals out
      for (int t = threadIdx.x; t < n; t += blockDim.x) {
        int run = 0;
        for (int ww = 0; ww < RPI_WARPS; ++ww) {
          int v = cnt[ww * n + t];
          cnt[ww * n + t] = run;
          run += v;
        }
        dir_counts[(int64_t)i * n + t] = run;
      }
      __syncthreads();
    }
  }
}

// pair_counts (column-major cell index a + b*n) and its exclusive scan; single block.
__global__ void k_pair_counts_scan(const int64_t* __restrict__ dir_counts, int n, int64_t* __restrict__ pair_counts,
                                   int64_t* __restrict__ pair_ptr) {
  __shared__ int64_t s_part[1024];
  const int64_t cells = (int64_t)n * n;
  const int tid = threadIdx.x, nt = blockDim.x;
  const int64_t per = (cells + nt - 1) / nt;
  const int64_t c0 = tid * per, c1 = min(cells, c0 + per);
  int64_t sum = 0;
  for (int64_t c = c0; c < c1; ++c) {
    int a = (int)(c % n), b = (int)(c / n);
    int64_t v = (a < b) ? dir_counts[(int64_t)a * n + b] + dir_counts[(int64_t)b * n + a] : 0;
    pair_counts[c] = v;
    sum += v;
  }
  s_part[tid] = sum;
  __syncthreads();
  if (tid == 0) {
    int64_t run = 0;
    for (int t = 0; t < nt; ++t) {
      int64_t v = s_part[t];
      s_part[t] = run;
      run += v;
    }
    pair_ptr[cells] = run;
  }
  __syncthreads();
  int64_t run = s_part[tid];
  for (int64_t c = c0; c < c1; ++c) {
    pair_ptr[c] = run;
    run += pair_counts[c];
  }
}

__global__ void k_scatter_rows(const int2* __restrict__ records,
                               const int32_t* __restrict__ img_of_row, const int64_t* __restrict__ img_off, int n,
                               int64_t F, const int64_t* __restrict__ dir_counts,
                               const int64_t* __restrict__ pair_ptr, const int64_t* __restrict__ rank,
                               uint32_t* __restrict__ rows) {
  int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= F) return;
  const int2 rec = records[q];
  const int t1 = rec.x;
  if (t1 <= 0) return;
  const int i = img_of_row[q], t = t1 - 1;
  const uint32_t li = (uint32_t)(q - img_off[i] + 1), lj = (uint32_t)rec.y;
  const int a = min(i, t), b = max(i, t);
  int64_t pos = pair_ptr[a + (int64_t)b * n] + rank[q];
  if (i > t) pos += dir_counts[(int64_t)a * n + b];  // the lower image's queries come first
  rows[2 * pos] = (i < t) ? li : lj;                 // featureMatchingGlobal.m:155-159
  rows[2 * pos + 1] = (i < t) ? lj : li;
}

// img_of_row is rebuilt here from img_off to keep the launcher signature small
__global__ void k_fill_img_of_row(const int64_t* __restrict__ img_off, int n, int32_t* __restrict__ img_of_row) {
  const int i = blockIdx.y;
  const int64_t b = img_off[i], e = img_off[i + 1];
  for (int64_t q = b + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < e; q += (int64_t)gridDim.x * blockDim.x)
    img_of_row[q] = i;
  (void)n;
}

int aps_k_fill_img_of_row(cudaStream_t s, const int64_t* img_off, int n, int64_t maxcount, int32_t* img_of_row) {
  if (n == 0 || maxcount == 0) return APS_OK;
  dim3 grid((unsigned)aps_min64(aps_ceil_div(maxcount, 256), 64), (unsigned)n);
  k_fill_img_of_row<<<grid, 256, 0, s>>>(img_off, n, img_of_row);
  APS_LAUNCHED();
  return APS_OK;
}

int aps_k_global_compact(cudaStream_t s, const int2* records,
                          const int32_t* img_of_row, const int64_t* img_off, int n, int64_t F, int64_t* dir_counts,
                          int64_t* pair_counts, int64_t* pair_ptr, int64_t* rank, uint32_t* rows) {
  if (n == 0) return APS_OK;
  if (n <= 1024)
    k_rank_per_image_mw<<<n, 32 * RPI_WARPS, (size_t)RPI_WARPS * n * sizeof(int), s>>>(records, img_off, n, dir_counts, rank);
  else
    k_rank_per_image<<<n, 32, (size_t)n * sizeof(int), s>>>(records, img_off, n, dir_counts, rank);
  APS_LAUNCHED();
  k_pair_counts_scan<<<1, 1024, 0, s>>>(dir_counts, n, pair_counts, pair_ptr);
  APS_LAUNCHED();
  if (F > 0) {
    k_scatter_rows<<<(unsigned)aps_ceil_div(F, 256), 256, 0, s>>>(records, img_of_row, img_off, n, F,
                                                                 dir_counts, pair_ptr, rank, rows);
    APS_LAUNCHED();
  }
  return APS_OK;
}

// ------------------------------------------------------------------------------------------------
// K5b over many independent image sets (aps_feature_matching_global_sets): the same cell order, but the cells of set s
// are its own n_s x n_s block at cell_off[s] -- sum(n_s^2) cells instead of (sum n_s)^2.  Records hold pooled image ids;
// a set's images are consecutive from set_img0[s], so local ids are pooled ids - set_img0[s].
struct SetTables {
  const int32_t* img_set;   // [images]: set of a pooled image
  const int32_t* set_img0;  // [sets]: first pooled image
  const int32_t* set_n;     // [sets]: images
  const int64_t* cell_off;  // [sets + 1]: first cell
};

__global__ void k_rank_per_image_sets(const int2* __restrict__ records, const int64_t* __restrict__ img_off,
                                      SetTables st, int64_t* __restrict__ dir_counts, int64_t* __restrict__ rank) {
  extern __shared__ int cnt[];  // [n of this image's set]
  const int i = blockIdx.x, lane = threadIdx.x;
  const int set = st.img_set[i], n = st.set_n[set], i0 = st.set_img0[set];
  for (int t = lane; t < n; t += 32) cnt[t] = 0;
  __syncwarp();
  const int64_t b = img_off[i], e = img_off[i + 1];
  for (int64_t base = b; base < e; base += 32) {
    const int64_t q = base + lane;
    const int t = (q < e) ? records[q].x : 0;
    const bool active = t > 0;
    const unsigned amask = __ballot_sync(0xffffffffu, active);
    int myrank = 0, cbase = 0;
    unsigned peers = 0;
    if (active) {
      peers = __match_any_sync(amask, t);
      cbase = cnt[t - 1 - i0];
      myrank = __popc(peers & ((1u << lane) - 1u));
    }
    __syncwarp();
    if (active) {
      rank[q] = (int64_t)cbase + myrank;
      if (myrank == 0) cnt[t - 1 - i0] = cbase + __popc(peers);
    }
    __syncwarp();
  }
  int64_t* dc = dir_counts + st.cell_off[set] + (int64_t)(i - i0) * n;
  for (int t = lane; t < n; t += 32) dc[t] = cnt[t];
}

// pair_counts of every set's block (column-major a + b*n inside it) and ONE exclusive scan over all cells; single block
__global__ void k_pair_counts_scan_sets(const int64_t* __restrict__ dir_counts, SetTables st, int nsets, int64_t cells,
                                        int64_t* __restrict__ pair_counts, int64_t* __restrict__ pair_ptr) {
  __shared__ int64_t s_part[1024];
  const int tid = threadIdx.x, nt = blockDim.x;
  const int64_t per = (cells + nt - 1) / nt;
  const int64_t c0 = min(cells, tid * per), c1 = min(cells, c0 + per);
  int lo = 0, hi = nsets;  // set holding cell c0: the last s with cell_off[s] <= c0
  while (hi - lo > 1) {
    const int mid = (lo + hi) / 2;
    if (st.cell_off[mid] <= c0) lo = mid;
    else hi = mid;
  }
  int64_t sum = 0;
  for (int64_t c = c0, set = lo; c < c1; ++c) {
    while (c >= st.cell_off[set + 1]) ++set;
    const int64_t n = st.set_n[set], cb = st.cell_off[set], l = c - cb;
    const int64_t a = l % n, b = l / n;
    const int64_t v = (a < b) ? dir_counts[cb + a * n + b] + dir_counts[cb + b * n + a] : 0;
    pair_counts[c] = v;
    sum += v;
  }
  s_part[tid] = sum;
  __syncthreads();
  if (tid == 0) {
    int64_t run = 0;
    for (int t = 0; t < nt; ++t) {
      int64_t v = s_part[t];
      s_part[t] = run;
      run += v;
    }
    pair_ptr[cells] = run;
  }
  __syncthreads();
  int64_t run = s_part[tid];
  for (int64_t c = c0; c < c1; ++c) {
    pair_ptr[c] = run;
    run += pair_counts[c];
  }
}

__global__ void k_scatter_rows_sets(const int2* __restrict__ records, const int32_t* __restrict__ img_of_row,
                                    const int64_t* __restrict__ img_off, SetTables st, int64_t F,
                                    const int64_t* __restrict__ dir_counts, const int64_t* __restrict__ pair_ptr,
                                    const int64_t* __restrict__ rank, uint32_t* __restrict__ rows) {
  int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= F) return;
  const int2 rec = records[q];
  if (rec.x <= 0) return;
  const int i = img_of_row[q], t = rec.x - 1, set = st.img_set[i], i0 = st.set_img0[set];
  const int64_t n = st.set_n[set], cb = st.cell_off[set];
  const uint32_t li = (uint32_t)(q - img_off[i] + 1), lj = (uint32_t)rec.y;
  const int64_t a = min(i, t) - i0, b = max(i, t) - i0;
  int64_t pos = pair_ptr[cb + a + b * n] + rank[q];
  if (i > t) pos += dir_counts[cb + a * n + b];  // the lower image's queries come first
  rows[2 * pos] = (i < t) ? li : lj;             // featureMatchingGlobal.m:155-159
  rows[2 * pos + 1] = (i < t) ? lj : li;
}

int aps_k_global_compact_sets(cudaStream_t s, const int2* records, const int32_t* img_of_row, const int64_t* img_off,
                              int nimg, int64_t F, const int32_t* img_set, const int32_t* set_img0, const int32_t* set_n,
                              const int64_t* cell_off, int nsets, int max_n, int64_t cells, int64_t* dir_counts,
                              int64_t* pair_counts, int64_t* pair_ptr, int64_t* rank, uint32_t* rows) {
  if (nsets == 0) return APS_OK;
  const SetTables st{img_set, set_img0, set_n, cell_off};
  const size_t smem = (size_t)max_n * sizeof(int);
  if (smem > 48 * 1024)
    APS_CUDA(cudaFuncSetAttribute(k_rank_per_image_sets, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  if (nimg > 0) {
    k_rank_per_image_sets<<<nimg, 32, smem, s>>>(records, img_off, st, dir_counts, rank);
    APS_LAUNCHED();
  }
  k_pair_counts_scan_sets<<<1, 1024, 0, s>>>(dir_counts, st, nsets, cells, pair_counts, pair_ptr);
  APS_LAUNCHED();
  if (F > 0) {
    k_scatter_rows_sets<<<(unsigned)aps_ceil_div(F, 256), 256, 0, s>>>(records, img_of_row, img_off, st, F, dir_counts,
                                                                       pair_ptr, rank, rows);
    APS_LAUNCHED();
  }
  return APS_OK;
}

// ------------------------------------------------------------------------------------------------
// Hamming 2-NN edge rows of the MEX contract (nearest2HammingExhaustiveMEX.cpp:42-45, 71-74).
__global__ void k_hamming2_finalize(int64_t N1, int64_t N2, int nb, const uint32_t* __restrict__ idx_k2,
                                    const float* __restrict__ dist_k2, uint32_t* __restrict__ idx2,
                                    float* __restrict__ d1, float* __restrict__ d2) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N1) return;
  if (N2 == 0) {
    idx2[i] = 0;
    d1[i] = CUDART_NAN_F;
    d2[i] = CUDART_NAN_F;
    return;
  }
  idx2[i] = idx_k2[2 * i];
  d1[i] = dist_k2[2 * i];
  d2[i] = (N2 == 1 || idx_k2[2 * i + 1] == 0u) ? (float)(nb * 8) : dist_k2[2 * i + 1];
}

int aps_k_hamming2_finalize(cudaStream_t s, int64_t N1, int64_t N2, int nb, const uint32_t* idx_k2,
                            const float* dist_k2, uint32_t* idx2, float* d1, float* d2) {
  if (N1 == 0) return APS_OK;
  k_hamming2_finalize<<<(unsigned)aps_ceil_div(N1, 256), 256, 0, s>>>(N1, N2, nb, idx_k2, dist_k2, idx2, d1, d2);
  APS_LAUNCHED();
  return APS_OK;
}

// SSD 2-NN from the k=2 search (matchFeaturesScratch.m:356-362): missing second -> +inf already.
__global__ void k_split_k2(int64_t N1, const uint32_t* __restrict__ idx_k2, const float* __restrict__ dist_k2,
                           uint32_t* __restrict__ idx2, float* __restrict__ d1, float* __restrict__ d2) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N1) return;
  idx2[i] = idx_k2[2 * i];
  d1[i] = dist_k2[2 * i];
  d2[i] = dist_k2[2 * i + 1];
}

int aps_k_split_k2(cudaStream_t s, int64_t N1, const uint32_t* idx_k2, const float* dist_k2, uint32_t* idx2,
                   float* d1, float* d2) {
  if (N1 == 0) return APS_OK;
  k_split_k2<<<(unsigned)aps_ceil_div(N1, 256), 256, 0, s>>>(N1, idx_k2, dist_k2, idx2, d1, d2);
  APS_LAUNCHED();
  return APS_OK;
}

// ------------------------------------------------------------------------------------------------
// matchFeaturesScratch.m:169-211 for one (query image, train image) pair.
//   key = (order-preserving bits of dBest) << 32 | (query index)  -> uniqueness = atomicMin per train
//   index (smallest d, ties -> lowest query index: equivalent to the reference's stable sort + greedy
//   accept because every query occurs once), output order = ascending key.
__device__ __forceinline__ uint32_t f32_order_bits(float f) {
  uint32_t b = __float_as_uint(f);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float f32_from_order_bits(uint32_t o) {
  uint32_t b = (o & 0x80000000u) ? (o & 0x7fffffffu) : ~o;
  return __uint_as_float(b);
}

__global__ void k_pair_keys(const uint32_t* __restrict__ idx2, const float* __restrict__ d1,
                            const float* __restrict__ d2, int64_t N1, int is_binary, int nbits,
                            double match_threshold, double max_ratio, int unique,
                            unsigned long long* __restrict__ best_by_train, unsigned long long* __restrict__ keys) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N1) return;
  bool keep;
  float dB;
  if (is_binary) {
    float s = d2[i];
    if (!isfinite(s) || s == 0.0f) s = (float)nbits;                                // :318
    dB = __fmul_rn(__fdiv_rn(d1[i], (float)nbits), 100.0f);                         // :120
    float dS = __fmul_rn(__fdiv_rn(s, (float)nbits), 100.0f);                       // :121
    float rhs = __fmul_rn((float)max_ratio, dS);                                    // :171 (single arithmetic)
    keep = (dB <= rhs) && (dB <= (float)match_threshold) && isfinite(dB) && isfinite(dS);
  } else {
    dB = d1[i];
    double b = (double)d1[i], sd = (double)d2[i];
    double r2 = max_ratio * max_ratio;                                              // :173
    keep = (b <= r2 * sd) && (b <= match_threshold) && isfinite(b) && isfinite(sd); // :174-178
  }
  unsigned long long key = ~0ull;
  if (keep) {
    // Unique: order by (d, query) ; otherwise keep the original query order (:208-209)
    key = unique ? (((unsigned long long)f32_order_bits(dB) << 32) | (unsigned long long)(uint32_t)i)
                 : (((unsigned long long)(uint32_t)i << 32) | (unsigned long long)f32_order_bits(dB));
    if (unique) atomicMin(&best_by_train[idx2[i] - 1], key);
  }
  keys[i] = key;
}

__global__ void k_pair_collect(const uint32_t* __restrict__ idx2, int64_t N1, int unique,
                               const unsigned long long* __restrict__ best_by_train,
                               const unsigned long long* __restrict__ keys, int32_t* __restrict__ count,
                               unsigned long long* __restrict__ winners) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  bool win = false;
  unsigned long long key = ~0ull;
  if (i < N1) {
    key = keys[i];
    win = key != ~0ull && (!unique || best_by_train[idx2[i] - 1] == key);
  }
  unsigned m = __ballot_sync(0xffffffffu, win);
  int base = 0;
  if ((threadIdx.x & 31) == 0 && m) base = atomicAdd(count, __popc(m));
  base = __shfl_sync(0xffffffffu, base, 0);
  if (win) winners[base + __popc(m & ((1u << (threadIdx.x & 31)) - 1u))] = key;
}

// rank-by-counting: winners are unique keys, rank = #smaller keys.  O(W^2) compares on a list that
// lives in shared-memory tiles -- negligible next to the N1*N2*D matching work of the same pair.
__global__ void k_pair_rank_emit(const unsigned long long* __restrict__ winners, const int32_t* __restrict__ count,
                                 const uint32_t* __restrict__ idx2, int unique, uint32_t* __restrict__ matches,
                                 double* __restrict__ metric) {
  __shared__ unsigned long long tile[1024];
  const int W = *count;
  for (int w0 = blockIdx.x * blockDim.x; w0 < W; w0 += gridDim.x * blockDim.x) {
    const int w = w0 + threadIdx.x;
    const unsigned long long mine = (w < W) ? winners[w] : ~0ull;
    int r = 0;
    for (int t0 = 0; t0 < W; t0 += 1024) {
      __syncthreads();
      for (int t = threadIdx.x; t < 1024; t += blockDim.x) tile[t] = (t0 + t < W) ? winners[t0 + t] : ~0ull;
      __syncthreads();
      const int nt = min(1024, W - t0);
      for (int t = 0; t < nt; ++t) r += (tile[t] < mine);
    }
    if (w < W) {
      const uint32_t lo = (uint32_t)(mine & 0xffffffffull), hi = (uint32_t)(mine >> 32);
      const uint32_t q = unique ? lo : hi;
      matches[2 * r] = q + 1;
      matches[2 * r + 1] = idx2[q];
      metric[r] = (double)f32_from_order_bits(unique ? hi : lo);
    }
  }
}

int aps_k_pair_filter_unique(cudaStream_t s, const uint32_t* idx2, const float* d1, const float* d2, int64_t N1,
                             int64_t N2, int is_binary, int nbits, double match_threshold, double max_ratio,
                             int unique, unsigned long long* best_by_train, unsigned long long* keys,
                             int32_t* count_dev, uint32_t* matches, double* metric) {
  if (N1 == 0 || N2 == 0) {
    APS_CUDA(cudaMemsetAsync(count_dev, 0, sizeof(int32_t), s));
    return APS_OK;
  }
  APS_CUDA(cudaMemsetAsync(best_by_train, 0xff, (size_t)N2 * sizeof(unsigned long long), s));
  APS_CUDA(cudaMemsetAsync(count_dev, 0, sizeof(int32_t), s));
  unsigned grid = (unsigned)aps_ceil_div(N1, 256);
  k_pair_keys<<<grid, 256, 0, s>>>(idx2, d1, d2, N1, is_binary, nbits, match_threshold, max_ratio, unique,
                                   best_by_train, keys);
  APS_LAUNCHED();
  // winners are written over best_by_train's tail?  No -- they get their own region: keys[N1..2*N1)
  unsigned long long* winners = keys + N1;
  k_pair_collect<<<grid, 256, 0, s>>>(idx2, N1, unique, best_by_train, keys, count_dev, winners);
  APS_LAUNCHED();
  unsigned rgrid = (unsigned)aps_min64(aps_ceil_div(N1, 256), 148);
  k_pair_rank_emit<<<rgrid, 256, 0, s>>>(winners, count_dev, idx2, unique, matches, metric);
  APS_LAUNCHED();
  return APS_OK;
}

// ------------------------------------------------------------------------------------------------
// K6  imageMatching.m:75-100 for every image set of a call.  Set b owns pooled images [set_img[b], set_img[b + 1]) and
// the n_b x n_b column-major block of cells at cell_off[b] (both tables [nsets + 1]); NULL tables = one set of n images.
// Stable descending order == rank by (value desc, column asc).
struct SelectSet {
  int64_t img0, cell0;
  int n;
};
// the set whose range [tab[b], tab[b + 1]) holds x (tab non-decreasing: empty sets are skipped)
__device__ __forceinline__ int select_set_of(const int64_t* __restrict__ tab, int nsets, int64_t x) {
  int lo = 0, hi = nsets;  // last b with tab[b] <= x
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (tab[mid] <= x) lo = mid; else hi = mid;
  }
  return lo;
}
__device__ __forceinline__ SelectSet select_set(const int64_t* __restrict__ set_img, const int64_t* __restrict__ cell_off,
                                                int nsets, int n, const int64_t* __restrict__ tab, int64_t x) {
  if (!set_img) return SelectSet{0, 0, n};
  const int b = select_set_of(tab, nsets, x);
  return SelectSet{set_img[b], cell_off[b], (int)(set_img[b + 1] - set_img[b])};
}

// one CTA per pooled image row: that row's partners ranked inside its own set's block
__global__ void k_select_rows(const int64_t* __restrict__ counts, int n, const int64_t* __restrict__ set_img,
                              const int64_t* __restrict__ cell_off, int nsets, int m, uint8_t* __restrict__ P) {
  const SelectSet S = select_set(set_img, cell_off, nsets, n, set_img, blockIdx.x);
  const int i = (int)(blockIdx.x - S.img0), nb = S.n;
  const int take = m < nb - 1 ? (m < 0 ? 0 : m) : nb - 1;
  const int64_t* C = counts + S.cell0;
  for (int j = threadIdx.x; j < nb; j += blockDim.x) {
    const int64_t sj = (i == j) ? 0 : C[i + (int64_t)j * nb] + C[j + (int64_t)i * nb];  // :82-83
    int r = 0;
    for (int c = 0; c < nb; ++c) {
      const int64_t sc = (i == c) ? 0 : C[i + (int64_t)c * nb] + C[c + (int64_t)i * nb];
      r += (sc > sj) || (sc == sj && c < j);
    }
    P[S.cell0 + i + (int64_t)j * nb] = r < take;  // :86-91
  }
}
__global__ void k_select_sym(const uint8_t* __restrict__ P, int n, const int64_t* __restrict__ set_img,
                             const int64_t* __restrict__ cell_off, int nsets, int64_t cells, uint8_t* __restrict__ cand) {
  int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= cells) return;
  const SelectSet S = select_set(set_img, cell_off, nsets, n, cell_off, c);
  const int64_t l = c - S.cell0;
  const int i = (int)(l % S.n), j = (int)(l / S.n);
  cand[c] = (i < j) && (P[S.cell0 + i + (int64_t)j * S.n] || P[S.cell0 + j + (int64_t)i * S.n]);  // :94-96
}

// find(candidatePairs) of every set in one CTA: ascending cell order == set-major, find() order inside a set.
// pairs_lin receives cell indices inside each set's block, set_pair_ptr [nsets + 1] the per-set offsets.
__global__ void __launch_bounds__(1024) k_select_compact(const uint8_t* __restrict__ cand, int64_t cells,
                                                         const int64_t* __restrict__ cell_off, int nsets,
                                                         int64_t* __restrict__ pairs_lin, int64_t* __restrict__ set_pair_ptr) {
  __shared__ int warp_cnt[32];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
  int64_t base = 0;
  for (int64_t c0 = 0; c0 < cells; c0 += blockDim.x) {
    const int64_t c = c0 + threadIdx.x;
    const bool sel = c < cells && cand[c];
    const unsigned bal = __ballot_sync(0xffffffffu, sel);
    if (lane == 0) warp_cnt[w] = __popc(bal);
    __syncthreads();
    int before = 0, tot = 0;
    for (int k = 0; k < nw; ++k) {
      before += k < w ? warp_cnt[k] : 0;
      tot += warp_cnt[k];
    }
    if (sel) pairs_lin[base + before + __popc(bal & ((1u << lane) - 1u))] = c;
    base += tot;
    __syncthreads();
  }
  for (int b = threadIdx.x; b <= nsets; b += blockDim.x) {  // pairs in cells before set b's block
    int64_t lo = 0, hi = base;
    while (lo < hi) {
      const int64_t mid = (lo + hi) >> 1;
      if (pairs_lin[mid] < cell_off[b]) lo = mid + 1; else hi = mid;
    }
    set_pair_ptr[b] = lo;
  }
  __syncthreads();
  for (int64_t k = threadIdx.x; k < base; k += blockDim.x)
    pairs_lin[k] -= cell_off[select_set_of(cell_off, nsets, pairs_lin[k])];
}

int aps_k_select_partners_sets(cudaStream_t s, const int64_t* counts, int n_rows, int64_t cells, const int64_t* set_img,
                               const int64_t* cell_off, int nsets, int m, uint8_t* cand) {
  if (n_rows == 0) return APS_OK;
  DevBuf<uint8_t> P;
  APS_TRY(P.alloc((size_t)cells, s));
  k_select_rows<<<n_rows, 128, 0, s>>>(counts, n_rows, set_img, cell_off, nsets, m, P.p);
  APS_LAUNCHED();
  k_select_sym<<<(unsigned)aps_ceil_div(cells, 256), 256, 0, s>>>(P.p, n_rows, set_img, cell_off, nsets, cells, cand);
  APS_LAUNCHED();
  return APS_OK;
}

int aps_k_select_partners(cudaStream_t s, const int64_t* counts_cm, int n, int m, uint8_t* cand_cm) {
  return aps_k_select_partners_sets(s, counts_cm, n, (int64_t)n * n, nullptr, nullptr, 1, m, cand_cm);
}

int aps_k_select_compact(cudaStream_t s, const uint8_t* cand, int64_t cells, const int64_t* cell_off, int nsets,
                         int64_t* pairs_lin, int64_t* set_pair_ptr) {
  k_select_compact<<<1, 1024, 0, s>>>(cand, cells, cell_off, nsets, pairs_lin, set_pair_ptr);
  APS_LAUNCHED();
  return APS_OK;
}
