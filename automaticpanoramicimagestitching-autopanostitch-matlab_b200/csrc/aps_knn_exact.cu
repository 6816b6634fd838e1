// aps_knn_exact.cu -- K2f: exact float kNN on CUDA cores.
//
// Role: (1) the provably-exact fallback for query rows whose tensor-core candidate set could not be
// proven complete (aps_rerank.cu), (2) the search engine for shapes the tcgen05 kernel does not
// take (D > 128, tiny problems), (3) nearest2SSDExhaustive's arithmetic.
//
// Replaces  cv::flann::Index::knnSearch behind PP/mex/flann_knn.cpp:229-234 (metric 0: squared L2 in
//           the order of FLANN's L2 functor, so distances are bit-identical to OpenCV's) and
//           PP/featureMatching/matchFeaturesScratch.m:351-358 (metric 1: (a2 + b2) - 2*G).
// Every float operation is an explicit _rn intrinsic: no FMA contraction, same bits as the oracle.
//
// Tiling: one CTA = RQ query rows (shared memory) x a stream of 256-row train tiles; thread t owns
// train row t of the tile and RQ running sums; the tile is staged through shared memory in chunks
// of 32 dimensions (row stride 36 floats -> conflict-free float4 reads).  Bound: FP32 pipe,
// 3 (L2) or 2 (SSD) FP32 instructions per dimension per pair.
#include <math_constants.h>

#include "aps_common.cuh"

namespace {

constexpr int RQ = 8;     // query rows per CTA == warps per CTA
constexpr int TJ = 256;   // train rows per tile == threads per CTA
constexpr int DC = 32;    // dimensions per staged chunk
constexpr int TLD = DC + 4;

// SETS: a group table drives the CTAs instead of (q0, nq, t0, t1): group g = rows [g.x, g.x + g.y) (g.y <= RQ) searched
// against train rows [g.z, g.w) only, neighbour indices 1-based over the whole matrix (number of groups: *nrows_dev when
// given -- a table built on the device -- else nq)
template <int METRIC, bool SETS = false>
__global__ void __launch_bounds__(TJ) k_knn_exact(const float* __restrict__ Q, const float* __restrict__ sqQ,
                                                   const int32_t* __restrict__ rows,
                                                   const int32_t* __restrict__ nrows_dev, int64_t q0, int64_t nq,
                                                   const float* __restrict__ T, const float* __restrict__ sqT,
                                                   int64_t t0, int64_t t1, int D, int k, int64_t out_row0,
                                                   uint32_t* __restrict__ idx, float* __restrict__ dist,
                                                   int nsplit, int64_t split_cap, uint32_t* __restrict__ pidx,
                                                   float* __restrict__ pdist, const int4* __restrict__ groups) {
  extern __shared__ __align__(16) float smem[];
  const int Dpad = (D + DC - 1) / DC * DC;
  float* qs = smem;                       // [RQ][Dpad]
  float* ts = qs + RQ * Dpad;             // [TJ][TLD]
  float* sd = ts + TJ * TLD;              // [RQ][TJ]
  float* topd = sd + RQ * TJ;             // [RQ][APS_MAX_K]
  uint32_t* topi = (uint32_t*)(topd + RQ * APS_MAX_K);
  __shared__ int64_t s_row[RQ];

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int64_t total = rows ? (int64_t)(*nrows_dev) : nq;
  const int64_t ngroups = SETS ? total : (total + RQ - 1) / RQ;
  const int nfull = D / 4;  // full groups of four (FLANN functor), then a scalar tail
  // few rows (the fallback list): split the train range over `ns` CTAs per row group, merge afterwards
  const int ns = (!SETS && nsplit > 1 && total <= split_cap) ? nsplit : 1;
  const int64_t tiles_all = (t1 - t0 + TJ - 1) / TJ, tiles_per = (tiles_all + ns - 1) / ns;

  for (int64_t work = blockIdx.x; work < ngroups * ns; work += gridDim.x) {
    const int64_t grp = work / ns;
    const int sp = (int)(work - grp * ns);
    int4 g = make_int4(0, 0, 0, 0);
    if (SETS) {
      g = groups[grp];
      t0 = g.z;
      t1 = g.w;
    }
    const int64_t ts0 = t0 + (int64_t)sp * tiles_per * TJ;
    const int64_t ts1 = SETS ? t1 : min(t1, ts0 + tiles_per * TJ);
    const int64_t ibase = SETS ? 0 : t0;  // neighbour index = train row - ibase + 1
    __syncthreads();
    if (tid < RQ) {
      int64_t i = grp * RQ + tid;
      if (SETS) s_row[tid] = tid < g.y ? (int64_t)g.x + tid : -1;
      else s_row[tid] = (i < total) ? (rows ? (int64_t)rows[i] : q0 + i) : -1;
    }
    if (tid < RQ * APS_MAX_K) {
      topd[tid] = CUDART_INF_F;
      topi[tid] = 0u;
    }
    __syncthreads();
    for (int i = tid; i < RQ * Dpad; i += TJ) {
      int r = i / Dpad, c = i - r * Dpad;
      int64_t row = s_row[r];
      qs[i] = (row >= 0 && c < D) ? Q[row * D + c] : 0.f;
    }
    float a2[RQ];
#pragma unroll
    for (int r = 0; r < RQ; ++r) a2[r] = (METRIC == 1 && s_row[r] >= 0) ? sqQ[s_row[r]] : 0.f;

    for (int64_t j0 = ts0; j0 < ts1; j0 += TJ) {
      float acc[RQ];
#pragma unroll
      for (int r = 0; r < RQ; ++r) acc[r] = 0.f;
      for (int d0 = 0; d0 < Dpad; d0 += DC) {
        __syncthreads();  // previous chunk consumed (also orders qs / sd use)
        for (int f = tid; f < TJ * (DC / 4); f += TJ) {
          int jr = f / (DC / 4), c4 = (f - jr * (DC / 4)) * 4;
          int64_t j = j0 + jr;
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
          if (j < t1) {
            const float* src = T + j * D + d0 + c4;
            if (d0 + c4 + 3 < D && (D & 3) == 0) {
              v = *reinterpret_cast<const float4*>(src);
            } else {
              if (d0 + c4 + 0 < D) v.x = src[0];
              if (d0 + c4 + 1 < D) v.y = src[1];
              if (d0 + c4 + 2 < D) v.z = src[2];
              if (d0 + c4 + 3 < D) v.w = src[3];
            }
          }
          *reinterpret_cast<float4*>(ts + jr * TLD + c4) = v;
        }
        __syncthreads();
#pragma unroll
        for (int g = 0; g < DC / 4; ++g) {
          const int gi = (d0 >> 2) + g;
          const float4 b = *reinterpret_cast<const float4*>(ts + tid * TLD + 4 * g);
          if (METRIC == 0) {
            if (gi < nfull) {
#pragma unroll
              for (int r = 0; r < RQ; ++r) {
                const float4 a = *reinterpret_cast<const float4*>(qs + r * Dpad + d0 + 4 * g);
                float e0 = __fsub_rn(a.x, b.x), e1 = __fsub_rn(a.y, b.y), e2 = __fsub_rn(a.z, b.z),
                      e3 = __fsub_rn(a.w, b.w);
                float s = __fadd_rn(__fmul_rn(e0, e0), __fmul_rn(e1, e1));
                s = __fadd_rn(s, __fmul_rn(e2, e2));
                s = __fadd_rn(s, __fmul_rn(e3, e3));
                acc[r] = __fadd_rn(acc[r], s);
              }
            } else if (4 * gi < D) {  // scalar tail of the functor (D % 4 != 0)
              const float bb[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
              for (int r = 0; r < RQ; ++r) {
                const float* a = qs + r * Dpad + d0 + 4 * g;
                for (int c = 0; c < 4 && 4 * gi + c < D; ++c) {
                  float e0 = __fsub_rn(a[c], bb[c]);
                  acc[r] = __fadd_rn(acc[r], __fmul_rn(e0, e0));
                }
              }
            }
          } else {
            if (4 * gi < D) {  // padded dimensions would add +0 products: harmless, but skip
#pragma unroll
              for (int r = 0; r < RQ; ++r) {
                const float4 a = *reinterpret_cast<const float4*>(qs + r * Dpad + d0 + 4 * g);
                float s = __fadd_rn(acc[r], __fmul_rn(a.x, b.x));
                s = __fadd_rn(s, __fmul_rn(a.y, b.y));
                s = __fadd_rn(s, __fmul_rn(a.z, b.z));
                acc[r] = __fadd_rn(s, __fmul_rn(a.w, b.w));
              }
            }
          }
        }
      }
      // distances of (query r, train j0+tid)
      const int64_t j = j0 + tid;
      const bool valid = j < t1;
      float b2 = (METRIC == 1 && valid) ? sqT[j] : 0.f;
#pragma unroll
      for (int r = 0; r < RQ; ++r) {
        float v = acc[r];
        if (METRIC == 1) v = __fsub_rn(__fadd_rn(a2[r], b2), __fmul_rn(2.0f, acc[r]));
        sd[r * TJ + tid] = valid ? v : CUDART_INF_F;
      }
      __syncthreads();
      // warp w merges the tile into query row w's ascending top-k (ascending j => ties keep the lower index)
      {
        const int r = warp;
        float worst = topd[r * APS_MAX_K + k - 1];
        for (int i = 0; i < TJ / 32; ++i) {
          const float v = sd[r * TJ + lane + 32 * i];
          unsigned ballot = __ballot_sync(0xffffffffu, v < worst);
          while (ballot) {
            const int l = __ffs(ballot) - 1;
            const float vl = __shfl_sync(0xffffffffu, v, l);
            if (lane == 0 && vl < worst) {
              int p = k - 1;
              while (p > 0 && vl < topd[r * APS_MAX_K + p - 1]) {
                topd[r * APS_MAX_K + p] = topd[r * APS_MAX_K + p - 1];
                topi[r * APS_MAX_K + p] = topi[r * APS_MAX_K + p - 1];
                --p;
              }
              topd[r * APS_MAX_K + p] = vl;
              topi[r * APS_MAX_K + p] = (uint32_t)(j0 + 32 * i + l - ibase + 1);
            }
            __syncwarp();
            worst = topd[r * APS_MAX_K + k - 1];
            ballot &= ~(1u << l);
            ballot &= __ballot_sync(0xffffffffu, v < worst);
          }
        }
      }
    }
    __syncthreads();
    if (lane < k && s_row[warp] >= 0) {
      if (ns == 1) {
        int64_t o = (s_row[warp] - out_row0) * k + lane;
        idx[o] = topi[warp * APS_MAX_K + lane];
        dist[o] = topd[warp * APS_MAX_K + lane];
      } else {
        int64_t o = ((grp * RQ + warp) * ns + sp) * k + lane;
        pidx[o] = topi[warp * APS_MAX_K + lane];
        pdist[o] = topd[warp * APS_MAX_K + lane];
      }
    }
  }
}

// merges the `ns` (<= 128) partial ascending lists of every row (ties -> lower index): one WARP per row, lane l owns
// the lists l, l+32, l+64, l+96; per output rank a shuffle arg-min over the lanes' best heads
__global__ void k_knn_exact_merge(const int32_t* __restrict__ rows, const int32_t* __restrict__ nrows_dev, int64_t q0,
                                  int64_t nq, int k, int nsplit, int64_t split_cap, const uint32_t* __restrict__ pidx,
                                  const float* __restrict__ pdist, int64_t out_row0, uint32_t* __restrict__ idx,
                                  float* __restrict__ dist) {
  const int64_t total = rows ? (int64_t)(*nrows_dev) : nq;
  if (!(nsplit > 1 && total <= split_cap)) return;
  const int lane = threadIdx.x & 31;
  const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (i >= total) return;  // warp-uniform
  const int64_t row = rows ? (int64_t)rows[i] : q0 + i;
  int head[4] = {0, 0, 0, 0};
  for (int c = 0; c < k; ++c) {
    float bd = CUDART_INF_F;  // every stored candidate has a finite distance: +inf == "no head left"
    uint32_t bi = 0xffffffffu;
    int bq = 0;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int sp = lane + 32 * q;
      if (sp < nsplit && head[q] < k) {
        const int64_t o = (i * nsplit + sp) * k + head[q];
        const uint32_t ci = pidx[o];
        if (ci != 0u) {
          const float cd = pdist[o];
          if (cd < bd || (cd == bd && ci < bi)) {
            bd = cd;
            bi = ci;
            bq = q;
          }
        }
      }
    }
    float wd = bd;
    uint32_t wi = bi;
    int wl = lane;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      const float od = __shfl_xor_sync(0xffffffffu, wd, off);
      const uint32_t oi = __shfl_xor_sync(0xffffffffu, wi, off);
      const int ol = __shfl_xor_sync(0xffffffffu, wl, off);
      if (od < wd || (od == wd && oi < wi)) {
        wd = od;
        wi = oi;
        wl = ol;
      }
    }
    const bool found = wi != 0xffffffffu;
    if (found && lane == wl) {
#pragma unroll
      for (int q = 0; q < 4; ++q) head[q] += (q == bq) ? 1 : 0;
    }
    if (lane == 0) {
      idx[(row - out_row0) * k + c] = found ? wi : 0u;
      dist[(row - out_row0) * k + c] = found ? wd : CUDART_INF_F;
    }
  }
}

}  // namespace

int aps_k_knn_exact(cudaStream_t s, const float* Q, const float* sqQ, const int32_t* rows, const int32_t* nrows_dev,
                    int64_t q0, int64_t nq, const float* T, const float* sqT, int64_t t0, int64_t t1, int D,
                    int k, int metric, int64_t out_row0, uint32_t* idx, float* dist) {
  if (nq == 0) return APS_OK;
  const int Dpad = (D + DC - 1) / DC * DC;
  size_t smem = (size_t)(RQ * Dpad + TJ * TLD + RQ * TJ + 2 * RQ * APS_MAX_K) * sizeof(float);
  if (smem > 200 * 1024) {
    aps_set_error(APS_ERR_DIM, "", "descriptor dimension %d too large for the exact kernel", D);
    return APS_ERR_DIM;
  }
  int64_t groups = aps_ceil_div(nq, RQ);
  // a row LIST (device-side count, usually tiny): let up to 128 CTAs share each row group's train range -- the kernel
  // is latency bound per CTA (load chunk, sync, compute, sync), so a short list wants many short sweeps (27 rows of
  // C2: 0.46 ms with 32 splits, profiles/r2_ncu_history.txt)
  const int64_t split_cap = 2048;
  int nsplit = 1;
  if (rows) {
    const int64_t tiles = aps_ceil_div(t1 - t0, TJ);
    nsplit = (int)(tiles < 128 ? (tiles < 1 ? 1 : tiles) : 128);
  }
  DevBuf<uint32_t> pidx;
  DevBuf<float> pdist;
  if (nsplit > 1) {
    const int64_t prow = aps_min64(nq, split_cap) + RQ;
    APS_TRY(pidx.alloc((size_t)prow * nsplit * k, s));
    APS_TRY(pdist.alloc((size_t)prow * nsplit * k, s));
  }
  unsigned grid = (unsigned)(groups * nsplit < 148 * 4 ? groups * nsplit : 148 * 4);
  if (metric == 0) {
    APS_CUDA(cudaFuncSetAttribute(k_knn_exact<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_knn_exact<0><<<grid, TJ, smem, s>>>(Q, sqQ, rows, nrows_dev, q0, nq, T, sqT, t0, t1, D, k, out_row0, idx, dist,
                                          nsplit, split_cap, pidx.p, pdist.p, nullptr);
  } else {
    APS_CUDA(cudaFuncSetAttribute(k_knn_exact<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_knn_exact<1><<<grid, TJ, smem, s>>>(Q, sqQ, rows, nrows_dev, q0, nq, T, sqT, t0, t1, D, k, out_row0, idx, dist,
                                          nsplit, split_cap, pidx.p, pdist.p, nullptr);
  }
  APS_LAUNCHED();
  if (nsplit > 1) {
    k_knn_exact_merge<<<(unsigned)aps_ceil_div(aps_min64(nq, split_cap), 4), 128, 0, s>>>(
        rows, nrows_dev, q0, nq, k, nsplit, split_cap, pidx.p, pdist.p, out_row0, idx, dist);
    APS_LAUNCHED();
  }
  return APS_OK;
}

// Set-restricted search (global path, metric 0): every group of the table holds up to 8 query rows of ONE set and the
// train range of that set, so rows never see another set's rows.  One launch for all sets; the neighbour indices are
// 1-based rows of the whole matrix.  ngroups_dev != nullptr: the table holds *ngroups_dev groups (at most ngroups),
// written on the device (e.g. the rows a re-rank could not prove).  Per row the result equals a search of the set alone:
// the candidates are merged in ascending train order with ties to the lower index, whatever the tiling.
int aps_k_knn_exact_groups(cudaStream_t s, const float* X, const int4* d_groups, int64_t ngroups,
                           const int32_t* ngroups_dev, int D, int k, uint32_t* idx, float* dist) {
  if (ngroups == 0) return APS_OK;
  const int Dpad = (D + DC - 1) / DC * DC;
  size_t smem = (size_t)(RQ * Dpad + TJ * TLD + RQ * TJ + 2 * RQ * APS_MAX_K) * sizeof(float);
  if (smem > 200 * 1024) {
    aps_set_error(APS_ERR_DIM, "", "descriptor dimension %d too large for the exact kernel", D);
    return APS_ERR_DIM;
  }
  const unsigned grid = (unsigned)(ngroups < 148 * 4 ? ngroups : 148 * 4);
  APS_CUDA(cudaFuncSetAttribute(k_knn_exact<0, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_knn_exact<0, true><<<grid, TJ, smem, s>>>(X, nullptr, ngroups_dev, ngroups_dev, 0, ngroups, X, nullptr, 0, 0, D, k,
                                              0, idx, dist, 1, 0, nullptr, nullptr, d_groups);
  APS_LAUNCHED();
  return APS_OK;
}
