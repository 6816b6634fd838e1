// aps_hamming.cu -- K4: exact Hamming kNN for packed binary descriptors (ORB 32 B, BRISK 64 B).
//
// Replaces  cv::BFMatcher(NORM_HAMMING).knnMatch behind PP/mex/flann_knn.cpp:199-223 (k = input.k)
//           and the triple loop of PP/mex/nearest2HammingExhaustiveMEX.cpp:50-79 /
//           PP/mex/nearest2HammingExhaustiveOMPMEX.cpp:52-82 (k = 2: best = first minimum, second =
//           2nd smallest value with multiplicity).
//
// Mapping: one thread = one query descriptor held in registers (NW x uint4); a CTA of 256 queries
// streams the train set through shared memory in 512-row tiles loaded with 128-bit coalesced
// loads; every thread reads the same train row (shared-memory broadcast), XOR + __popc, and keeps
// an ascending top-K in registers (scan order is ascending train index, strict '<' => ties keep the
// lower index, as BFMatcher and the MEX do).  Integer work on CUDA cores -- deliberately not
// reshaped into a GEMM.  Bound: POPC + LOP3 issue (carry-save adders: 5 popc + 14 lop3 per 256-bit pair); operand bytes come from
// shared memory, HBM sees each train row once per CTA (L2-resident for F <= ~10^6 rows).
#include <math_constants.h>

#include "aps_common.cuh"
#include "aps_hamming.cuh"

namespace {

constexpr int HQ = 256;  // queries per CTA
constexpr int HT = 512;  // train rows per shared-memory tile

// SETS: CTA b takes group groups[b] = rows [g.x, g.x + g.y) (g.y <= HQ) searched against train rows [g.z, g.w) only,
// neighbour indices 1-based over the whole matrix (q0, nq, t0, t1 unused)
template <int NW, int KT, bool SETS = false>
__global__ void __launch_bounds__(HQ) k_knn_hamming(const uint4* __restrict__ Q, int64_t q0, int64_t nq,
                                                     const uint4* __restrict__ T, int64_t t0, int64_t t1, int k,
                                                     int64_t out_row0, uint32_t* __restrict__ idx,
                                                     float* __restrict__ dist, const int4* __restrict__ groups) {
  __shared__ uint4 ts[HT * NW];
  const int tid = threadIdx.x;
  int64_t q, ibase = t0;  // neighbour index = train row - ibase + 1
  bool qvalid;
  if (SETS) {
    const int4 g = groups[blockIdx.x];
    q = (int64_t)g.x + tid;
    qvalid = tid < g.y;
    t0 = g.z;
    t1 = g.w;
    ibase = 0;
  } else {
    q = q0 + (int64_t)blockIdx.x * HQ + tid;
    qvalid = q < q0 + nq;
  }
  uint4 a[NW];
#pragma unroll
  for (int w = 0; w < NW; ++w) a[w] = qvalid ? Q[q * NW + w] : make_uint4(0, 0, 0, 0);
  int bd[KT];
  uint32_t bi[KT];
#pragma unroll
  for (int c = 0; c < KT; ++c) {
    bd[c] = 0x7fffffff;
    bi[c] = 0u;
  }
  for (int64_t j0 = t0; j0 < t1; j0 += HT) {
    const int nj = (int)min((int64_t)HT, t1 - j0);
    __syncthreads();
    for (int f = tid; f < nj * NW; f += HQ) ts[f] = T[j0 * NW + f];
    __syncthreads();
#pragma unroll 4
    for (int j = 0; j < nj; ++j) {
      const int h = hamming_words<NW>(a, ts + j * NW);
      if (h < bd[KT - 1]) {
        bd[KT - 1] = h;
        bi[KT - 1] = (uint32_t)(j0 + j - ibase + 1);
#pragma unroll
        for (int p = KT - 1; p > 0; --p) {
          if (bd[p] < bd[p - 1]) {
            int td = bd[p]; bd[p] = bd[p - 1]; bd[p - 1] = td;
            uint32_t ti = bi[p]; bi[p] = bi[p - 1]; bi[p - 1] = ti;
          }
        }
      }
    }
  }
  if (qvalid) {
#pragma unroll
    for (int c = 0; c < KT; ++c)
      if (c < k) {
        int64_t o = (q - out_row0) * k + c;
        idx[o] = bi[c];
        dist[o] = bi[c] ? (float)bd[c] : CUDART_INF_F;  // flann_knn.cpp:216-219
      }
  }
}

template <int NW>
int launch_nw(cudaStream_t s, const uint8_t* Q, int64_t q0, int64_t nq, const uint8_t* T, int64_t t0, int64_t t1,
              int k, int64_t out_row0, uint32_t* idx, float* dist) {
  unsigned grid = (unsigned)aps_ceil_div(nq, HQ);
  const uint4* q4 = (const uint4*)Q;
  const uint4* t4 = (const uint4*)T;
  if (k <= 2)
    k_knn_hamming<NW, 2><<<grid, HQ, 0, s>>>(q4, q0, nq, t4, t0, t1, k, out_row0, idx, dist, nullptr);
  else if (k <= 4)
    k_knn_hamming<NW, 4><<<grid, HQ, 0, s>>>(q4, q0, nq, t4, t0, t1, k, out_row0, idx, dist, nullptr);
  else if (k <= 8)
    k_knn_hamming<NW, 8><<<grid, HQ, 0, s>>>(q4, q0, nq, t4, t0, t1, k, out_row0, idx, dist, nullptr);
  else if (k <= 16)
    k_knn_hamming<NW, 16><<<grid, HQ, 0, s>>>(q4, q0, nq, t4, t0, t1, k, out_row0, idx, dist, nullptr);
  else
    k_knn_hamming<NW, 32><<<grid, HQ, 0, s>>>(q4, q0, nq, t4, t0, t1, k, out_row0, idx, dist, nullptr);
  APS_LAUNCHED();
  return APS_OK;
}

template <int NW, int KT>
void launch_groups(cudaStream_t s, const uint8_t* X, const int4* groups, int64_t ngroups, int k, uint32_t* idx,
                   float* dist) {
  const uint4* x4 = (const uint4*)X;
  k_knn_hamming<NW, KT, true><<<(unsigned)ngroups, HQ, 0, s>>>(x4, 0, 0, x4, 0, 0, k, 0, idx, dist, groups);
}

template <int NW>
int launch_groups_nw(cudaStream_t s, const uint8_t* X, const int4* groups, int64_t ngroups, int k, uint32_t* idx,
                     float* dist) {
  if (k <= 2) launch_groups<NW, 2>(s, X, groups, ngroups, k, idx, dist);
  else if (k <= 4) launch_groups<NW, 4>(s, X, groups, ngroups, k, idx, dist);
  else if (k <= 8) launch_groups<NW, 8>(s, X, groups, ngroups, k, idx, dist);
  else if (k <= 16) launch_groups<NW, 16>(s, X, groups, ngroups, k, idx, dist);
  else launch_groups<NW, 32>(s, X, groups, ngroups, k, idx, dist);
  APS_LAUNCHED();
  return APS_OK;
}

}  // namespace

// Set-restricted search of the pooled rows X (padded to nb16): one launch, one CTA per group of up to 256 rows of one
// set, each against its own set's rows (aps_k_knn_exact_groups' table with HQ-row groups).
int aps_k_knn_hamming_groups(cudaStream_t s, const uint8_t* X, const int4* d_groups, int64_t ngroups, int nb16, int k,
                             uint32_t* idx, float* dist) {
  if (ngroups == 0) return APS_OK;
  switch (nb16 / 16) {
    case 1: return launch_groups_nw<1>(s, X, d_groups, ngroups, k, idx, dist);
    case 2: return launch_groups_nw<2>(s, X, d_groups, ngroups, k, idx, dist);
    case 3: return launch_groups_nw<3>(s, X, d_groups, ngroups, k, idx, dist);
    case 4: return launch_groups_nw<4>(s, X, d_groups, ngroups, k, idx, dist);
    default:
      aps_set_error(APS_ERR_DIM, "hamm2nn:cols", "binary descriptors wider than 64 bytes are not supported (%d)", nb16);
      return APS_ERR_DIM;
  }
}
int aps_k_knn_hamming_group_rows() { return HQ; }

// Q, T: rows padded to nb16 = multiple of 16 bytes (zero padded: pads XOR to zero), 16-byte aligned.
int aps_k_knn_hamming(cudaStream_t s, const uint8_t* Q, int64_t q0, int64_t nq, const uint8_t* T, int64_t t0,
                      int64_t t1, int nb16, int k, int64_t out_row0, uint32_t* idx, float* dist) {
  if (nq == 0) return APS_OK;
  switch (nb16 / 16) {
    case 1: return launch_nw<1>(s, Q, q0, nq, T, t0, t1, k, out_row0, idx, dist);
    case 2: return launch_nw<2>(s, Q, q0, nq, T, t0, t1, k, out_row0, idx, dist);
    case 3: return launch_nw<3>(s, Q, q0, nq, T, t0, t1, k, out_row0, idx, dist);
    case 4: return launch_nw<4>(s, Q, q0, nq, T, t0, t1, k, out_row0, idx, dist);
    default:
      aps_set_error(APS_ERR_DIM, "hamm2nn:cols", "binary descriptors wider than 64 bytes are not supported (%d)", nb16);
      return APS_ERR_DIM;
  }
}
