// aps_pair_screen.cu -- pairwise path, stage 1: tensor-core SCREEN of every (query row, train image).
//
// Replaces, for the image pairs that cannot produce a match, the whole of
//     PP/featureMatching/matchFeaturesScratch.m:343-358 (SSD by GEMM, two min passes) + :169-178 (ratio / threshold).
// The reference keeps a query only if  d1 <= MaxRatio^2 * d2  and  d1 <= MatchThreshold  (:174-178).  In a multi-
// panorama set almost every (query, train image) fails that test by a wide margin (C5: 99.7 %), so it is enough to
// BOUND d1 from below and d2 from above:
//     dot(q, j)  = a_q . b_j                         fp16 operands, tcgen05.mma kind::f16 with FP16 accumulators in TMEM
//     b1 >= b2   = the two largest of the 8 class maxima (columns by  column mod 8): two DISTINCT train rows
//     d1 >= |a|^2 + min_j |b_j|^2 - 2 (b1 + e)  ,  d2 <= |a|^2 + max_j |b_j|^2 - 2 (b2 - e)
// (e = bound of the fp16 operand / accumulation error, aps_k_pair_screen_eps).  A row whose bounds already violate
// the test is rejected without ever computing an exact distance or an index; image pairs in which some row survives go
// through the exact pipeline (aps_knn_tc.cu + aps_rerank.cu + k_pair_exact2), so the match lists stay bit-identical to
// the oracle's.  Nothing index-like is tracked here, which is what makes the epilogue cheap: the packed FP16
// accumulators are read with tcgen05.ld (two scores per register) and folded with HMNMX2 -- 0.5 instructions per
// score instead of ~7.6 in the selecting epilogue (profiles/r1_ncu_k_knn_tc_pairwise.txt: ALU-pipe bound).
//
// CTA = 352 threads, persistent over work units (one unit = 256 query rows of image i x all tiles of image j):
//   warp 0   : TMA producer (A pair double-buffered across units, B ring)
//   warps 1-2: one single-thread tcgen05.mma issuer per 128-row block
//   warps 3-10: epilogue, thread == query row, 2 accumulator phases of 128 TMEM columns per row block; the f16
//              accumulators are read with tcgen05.ld .pack::16b (two scores per register)
// Roofline: tensor pipe (2*D FLOP per pair); operands stream from L2 (consecutive units share the train image).
#include <cuda_fp16.h>

#include "aps_tc_ptx.cuh"

namespace {
using namespace aps_tc;

constexpr int TM = 128, TN = 128, RB = 2;
constexpr int ACC_PHASES = 2;                 // accumulator slots per row block
constexpr int ACC_COLS = TN;                  // an f16 accumulator still owns a 32-bit TMEM column (16 bits used);
                                              // tcgen05.ld .pack::16b packs two adjacent columns into one register
constexpr int NUM_EPI_WARPS = 4 * RB;
constexpr int FIRST_EPI_WARP = 1 + RB;
constexpr int NUM_THREADS = 32 * (FIRST_EPI_WARP + NUM_EPI_WARPS);
constexpr int MAX_B_STAGES = 8;
constexpr uint32_t NEG2 = 0xFBFFFBFFu;        // (-65504, -65504): below every finite dot

struct Bars {
  uint64_t b_full[MAX_B_STAGES], b_empty[MAX_B_STAGES];
  uint64_t a_full[2], a_empty[2];
  uint64_t acc_full[ACC_PHASES * RB], acc_empty[ACC_PHASES * RB];
  uint32_t tmem_base, pad;
};

struct SParams {
  const aps_tc_unit* units;
  int64_t n_units;
  int dp, b_stages, a_bufs;
  uint32_t* out;        // [entries] packed half2 (b1, b2)
  uint32_t* dump;       // tests: raw accumulator registers [entries][dump_tiles][64], else nullptr
  int dump_tiles;
  uint32_t idesc;       // tcgen05 instruction descriptor (kind::f16: F16 operands, F16 accumulators)
};

// 64 TMEM columns of 16-bit accumulators -> 32 registers of two packed fp16 (columns 2j, 2j+1 -> register j)
static __device__ __forceinline__ void tmem_ld64p(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.pack::16b.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
static __device__ __forceinline__ void tmem_wait_ld2(uint32_t (&a)[32], uint32_t (&b)[32]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(a[0]), "+r"(a[1]), "+r"(a[2]), "+r"(a[3]), "+r"(a[4]), "+r"(a[5]), "+r"(a[6]), "+r"(a[7]),
                 "+r"(a[8]), "+r"(a[9]), "+r"(a[10]), "+r"(a[11]), "+r"(a[12]), "+r"(a[13]), "+r"(a[14]), "+r"(a[15]),
                 "+r"(a[16]), "+r"(a[17]), "+r"(a[18]), "+r"(a[19]), "+r"(a[20]), "+r"(a[21]), "+r"(a[22]), "+r"(a[23]),
                 "+r"(a[24]), "+r"(a[25]), "+r"(a[26]), "+r"(a[27]), "+r"(a[28]), "+r"(a[29]), "+r"(a[30]), "+r"(a[31])
               :
               : "memory");
  asm volatile("" : "+r"(b[0]), "+r"(b[1]), "+r"(b[2]), "+r"(b[3]), "+r"(b[4]), "+r"(b[5]), "+r"(b[6]), "+r"(b[7]),
                    "+r"(b[8]), "+r"(b[9]), "+r"(b[10]), "+r"(b[11]), "+r"(b[12]), "+r"(b[13]), "+r"(b[14]), "+r"(b[15]),
                    "+r"(b[16]), "+r"(b[17]), "+r"(b[18]), "+r"(b[19]), "+r"(b[20]), "+r"(b[21]), "+r"(b[22]), "+r"(b[23]),
                    "+r"(b[24]), "+r"(b[25]), "+r"(b[26]), "+r"(b[27]), "+r"(b[28]), "+r"(b[29]), "+r"(b[30]), "+r"(b[31])
               :
               : "memory");
}
static __device__ __forceinline__ uint32_t hmax2u(uint32_t a, uint32_t b) {
  uint32_t d;
  asm("max.f16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b));
  return d;
}
static __device__ __forceinline__ uint32_t hmin2u(uint32_t a, uint32_t b) {
  uint32_t d;
  asm("min.f16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b));
  return d;
}

__global__ void __launch_bounds__(NUM_THREADS, 1)
k_pair_screen(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_t, const SParams P) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  const int a_bytes = TM * P.dp * 2, b_bytes = TN * P.dp * 2;
  uint8_t* smem_a = smem;                                      // a_bufs x RB x a_bytes
  uint8_t* smem_b = smem_a + P.a_bufs * RB * a_bytes;          // b_stages x b_bytes
  Bars* bars = (Bars*)(smem_b + P.b_stages * b_bytes);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ksl = P.dp / KSLAB, kst = P.dp / 16;
  const int NB = P.b_stages, NA = P.a_bufs;

  if (threadIdx.x == 0) {
    for (int i = 0; i < NB; ++i) { mbar_init(&bars->b_full[i], 1); mbar_init(&bars->b_empty[i], RB); }
    for (int i = 0; i < 2; ++i) { mbar_init(&bars->a_full[i], 1); mbar_init(&bars->a_empty[i], RB); }
    for (int i = 0; i < ACC_PHASES * RB; ++i) { mbar_init(&bars->acc_full[i], 1); mbar_init(&bars->acc_empty[i], 4); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&bars->tmem_base)), "r"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = bars->tmem_base;

  if (warp == 0) {
    // ===================================== TMA producer =====================================
    if (elect_one()) {
      uint32_t bs = 0, bph = 0, ucount = 0;
      for (int64_t u = blockIdx.x; u < P.n_units; u += gridDim.x, ++ucount) {
        const aps_tc_unit x = P.units[u];
        const uint32_t ab = ucount % NA, aph = (ucount / NA) & 1;
        mbar_wait_backoff(&bars->a_empty[ab], aph ^ 1);
        mbar_arrive_expect_tx(&bars->a_full[ab], (uint32_t)(RB * a_bytes));
        for (int r = 0; r < RB; ++r)
          for (int s = 0; s < ksl; ++s)
            tma_load_2d(smem_a + (ab * RB + r) * a_bytes + s * (TM * 128), &map_q, s * KSLAB, x.qrow0 + r * TM,
                        &bars->a_full[ab]);
        const int tl = x.t0 / TN, th = (x.t1 + TN - 1) / TN;
        for (int t = tl; t < th; ++t) {
          mbar_wait_backoff(&bars->b_empty[bs], bph ^ 1);
          mbar_arrive_expect_tx(&bars->b_full[bs], (uint32_t)b_bytes);
          for (int s = 0; s < ksl; ++s)
            tma_load_2d(smem_b + bs * b_bytes + s * (TN * 128), &map_t, s * KSLAB, t * TN, &bars->b_full[bs]);
          if (++bs == (uint32_t)NB) { bs = 0; bph ^= 1; }
        }
      }
    }
  } else if (warp <= RB) {
    // ===================================== MMA issuers =======================================
    // elect.sync instead of "lane == 0": the compiler then knows exactly one thread runs the loop and keeps the
    // descriptors in uniform registers (a lane-id guard costs a ~20-instruction R2UR waterfall per tcgen05.mma)
    if (elect_one()) {
      const int r = warp - 1;
      const uint32_t idesc = P.idesc;
      uint32_t bs = 0, bph = 0, tcount = 0, ucount = 0;
      for (int64_t u = blockIdx.x; u < P.n_units; u += gridDim.x, ++ucount) {
        const aps_tc_unit x = P.units[u];
        const uint32_t ab = ucount % NA, aph = (ucount / NA) & 1;
        const uint32_t a_addr = smem_u32(smem_a + (ab * RB + r) * a_bytes);
        mbar_wait(&bars->a_full[ab], aph);
        const int tl = x.t0 / TN, th = (x.t1 + TN - 1) / TN;
        for (int t = tl; t < th; ++t, ++tcount) {
          const uint32_t slot = (tcount % ACC_PHASES) * RB + r, acph = (tcount / ACC_PHASES) & 1;
          mbar_wait(&bars->acc_empty[slot], acph ^ 1);
          mbar_wait(&bars->b_full[bs], bph);
          tc_fence_after();
          const uint32_t b_addr = smem_u32(smem_b + bs * b_bytes);
          const uint32_t d_tmem = tmem_base + slot * ACC_COLS;
          for (int k = 0; k < kst; ++k) {
            const int slab = k >> 2, kin = k & 3;
            const uint64_t adesc = make_kmajor_sw128_desc(a_addr + slab * (TM * 128) + kin * 32);
            const uint64_t bdesc = make_kmajor_sw128_desc(b_addr + slab * (TN * 128) + kin * 32);
            umma_bf16(d_tmem, adesc, bdesc, idesc, k > 0 ? 1u : 0u);   // kind::f16; operand / accumulator types are in idesc
          }
          tc_commit(&bars->acc_full[slot]);
          tc_commit(&bars->b_empty[bs]);
          if (++bs == (uint32_t)NB) { bs = 0; bph ^= 1; }
        }
        tc_commit(&bars->a_empty[ab]);
      }
    }
  } else {
    // ===================================== epilogue =========================================
    const int quad = warp & 3;
    const int grp = (warp - FIRST_EPI_WARP) >> 2;   // row block of the unit
    const int row_in_tile = quad * 32 + lane;
    uint32_t tcount = 0;
    for (int64_t u = blockIdx.x; u < P.n_units; u += gridDim.x) {
      const aps_tc_unit x = P.units[u];
      const int tl = x.t0 / TN, th = (x.t1 + TN - 1) / TN;
      uint32_t m[4] = {NEG2, NEG2, NEG2, NEG2};   // class maxima: m[i].lo = columns == 2i (mod 8), m[i].hi = 2i+1 (mod 8)
      for (int t = tl; t < th; ++t, ++tcount) {
        const uint32_t slot = (tcount % ACC_PHASES) * RB + grp, acph = (tcount / ACC_PHASES) & 1;
        mbar_wait(&bars->acc_full[slot], acph);
        tc_fence_after();
        const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + slot * ACC_COLS;
        uint32_t va[32], vb[32];
        tmem_ld64p(taddr, va);
        tmem_ld64p(taddr + 64, vb);
        tmem_wait_ld2(va, vb);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&bars->acc_empty[slot]);   // registers hold the tile: the slot can be refilled
        if (P.dump) {
          const int64_t e = x.out_row + grp * TM + row_in_tile;
          if (x.qrow0 + grp * TM + row_in_tile < x.qend && t - tl < P.dump_tiles) {
            uint32_t* d = P.dump + (e * P.dump_tiles + (t - tl)) * 64;
#pragma unroll
            for (int j = 0; j < 32; ++j) { d[j] = va[j]; d[32 + j] = vb[j]; }
          }
        }
        const int lo = (t == tl) ? (x.t0 - t * TN) : 0, hi = (t == th - 1) ? (x.t1 - t * TN) : TN;
        if (lo > 0 || hi < TN) {   // first / last tile of the train image: foreign columns can never be a maximum
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const int c0 = 2 * j, c1 = 2 * j + 1;
            const uint32_t ma = ((c0 >= lo && c0 < hi) ? 0x0000FFFFu : 0u) | ((c1 >= lo && c1 < hi) ? 0xFFFF0000u : 0u);
            const uint32_t mb = ((c0 + 64 >= lo && c0 + 64 < hi) ? 0x0000FFFFu : 0u) | ((c1 + 64 >= lo && c1 + 64 < hi) ? 0xFFFF0000u : 0u);
            va[j] = (va[j] & ma) | (NEG2 & ~ma);
            vb[j] = (vb[j] & mb) | (NEG2 & ~mb);
          }
        }
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
          m[0] = hmax2u(m[0], hmax2u(va[j], vb[j]));
          m[1] = hmax2u(m[1], hmax2u(va[j + 1], vb[j + 1]));
          m[2] = hmax2u(m[2], hmax2u(va[j + 2], vb[j + 2]));
          m[3] = hmax2u(m[3], hmax2u(va[j + 3], vb[j + 3]));
        }
      }
      // two largest of the 8 class maxima (distinct classes => distinct train rows)
      uint32_t h01 = hmax2u(m[0], m[1]), l01 = hmin2u(m[0], m[1]);
      uint32_t h23 = hmax2u(m[2], m[3]), l23 = hmin2u(m[2], m[3]);
      uint32_t h = hmax2u(h01, h23), l = hmax2u(hmin2u(h01, h23), hmax2u(l01, l23));   // per half-lane: best, second
      const __half2 hh = *reinterpret_cast<__half2*>(&h), ll = *reinterpret_cast<__half2*>(&l);
      const float h0 = __low2float(hh), h1 = __high2float(hh), l0 = __low2float(ll), l1 = __high2float(ll);
      const float b1 = fmaxf(h0, h1);
      const float b2 = fmaxf(fminf(h0, h1), (h0 >= h1) ? l0 : l1);
      if (x.qrow0 + grp * TM + row_in_tile < x.qend) {
        const __half2 o = __floats2half2_rn(b1, b2);   // exact: both are fp16 values
        P.out[x.out_row + grp * TM + row_in_tile] = *reinterpret_cast<const uint32_t*>(&o);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}

// fp16 operand rows [F x Dp] (K-major, zero padded)
__global__ void k_prepare_operands_f16(const float* __restrict__ src, int64_t F, int D, int Dp, __half* __restrict__ xh) {
  const int chunks = Dp / 8;
  const int64_t total = F * chunks;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / chunks;
    const int c0 = (int)(i - r * chunks) * 8;
    __align__(16) __half v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = __float2half_rn(c0 + j < D ? src[r * D + c0 + j] : 0.0f);
    *reinterpret_cast<uint4*>(xh + r * Dp + c0) = *reinterpret_cast<const uint4*>(v);
  }
}

__global__ void k_fill_f32(float* __restrict__ dst, int64_t n, float v) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) dst[i] = v;
}

// per image: (min, max) of the squared row norms
__global__ void k_image_sq_bounds(const float* __restrict__ sq, const int64_t* __restrict__ start,
                                  const int64_t* __restrict__ count, float2* __restrict__ out) {
  const int i = blockIdx.x;
  float mn = 3.0e38f, mx = 0.f;
  for (int64_t r = start[i] + threadIdx.x; r < start[i] + count[i]; r += blockDim.x) {
    mn = fminf(mn, sq[r]);
    mx = fmaxf(mx, sq[r]);
  }
  __shared__ float smn[32], smx[32];
  for (int o = 16; o > 0; o >>= 1) {
    mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  }
  if ((threadIdx.x & 31) == 0) { smn[threadIdx.x >> 5] = mn; smx[threadIdx.x >> 5] = mx; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w) { mn = fminf(mn, smn[w]); mx = fmaxf(mx, smx[w]); }
    out[i] = make_float2(mn, mx);
  }
}

// units of the screen launch: pair p, 256-row block b
__global__ void k_make_units(const int32_t* __restrict__ qoff, const int32_t* __restrict__ qcnt,
                             const int32_t* __restrict__ toff, const int32_t* __restrict__ tcnt,
                             const int64_t* __restrict__ eoff, const int64_t* __restrict__ uoff, int npairs,
                             aps_tc_unit* __restrict__ units) {
  const int p = blockIdx.x;
  if (p >= npairs) return;
  const int64_t u0 = uoff[p], nu = uoff[p + 1] - u0;
  for (int64_t b = threadIdx.x; b < nu; b += blockDim.x) {
    aps_tc_unit u;
    u.qrow0 = qoff[p] + (int32_t)(b * RB * TM);
    u.qend = qoff[p] + qcnt[p];
    u.t0 = toff[p];
    u.t1 = toff[p] + tcnt[p];
    u.out_row = eoff[p] + b * RB * TM;
    units[u0 + b] = u;
  }
}

// decision: survivors per pair.  One block per pair.
__global__ void k_pair_screen_decide(const uint32_t* __restrict__ scr, const float* __restrict__ sq,
                                     const int32_t* __restrict__ qoff, const int32_t* __restrict__ qcnt,
                                     const int32_t* __restrict__ timg, const int64_t* __restrict__ eoff,
                                     const float2* __restrict__ img_bounds, const int32_t* __restrict__ flags,
                                     int Dp, double r2, double mt, int32_t* __restrict__ survivors) {
  const int p = blockIdx.x;
  const float2 bb = img_bounds[timg[p]];
  const float maxsq = fmaxf(__int_as_float(flags[2]), 1.0f);
  const double e = (double)aps_pair_screen_dot_eps(Dp) * (double)maxsq;
  int mine = 0;
  for (int r = threadIdx.x; r < qcnt[p]; r += blockDim.x) {
    const uint32_t v = scr[eoff[p] + r];
    const __half2 h = *reinterpret_cast<const __half2*>(&v);
    const double b1 = (double)__low2float(h), b2 = (double)__high2float(h);
    const double a2 = (double)sq[qoff[p] + r];
    const double lb1 = a2 + (double)bb.x - 2.0 * (b1 + e);   // exact d1 >= lb1
    const double ub2 = a2 + (double)bb.y - 2.0 * (b2 - e);   // exact d2 <= ub2
    const double slack = 1e-4 * (double)maxsq + 1e-6 * (fabs(lb1) + 1.0);
    const bool rej = (lb1 > r2 * ub2 + slack) || (lb1 > mt + slack);
    mine += !rej;
  }
  mine = __reduce_add_sync(0xffffffffu, mine);
  if ((threadIdx.x & 31) == 0 && mine) atomicAdd(&survivors[p], mine);
}

// ---- 'subsetpdist2' above the subset size: candB = randperm(N2, subset) (matchFeaturesScratch.m:391-392) -----------------
// Stand-in for MATLAB's generator: a keyed bijection of [0, N) (odd multiplications, xor-shifts and additions modulo a power
// of two, cycle-walked into range); candB[r] = perm(r), r = 0 .. subset-1: `subset` distinct rows in a pseudo-random order.
__device__ __forceinline__ uint32_t perm_in_range(uint32_t x, uint32_t N, uint64_t key) {
  int bits = 1;
  while ((1u << bits) < N && bits < 31) ++bits;
  const uint32_t mask = (bits >= 32) ? 0xffffffffu : ((1u << bits) - 1u);
  const uint32_t k0 = (uint32_t)key, k1 = (uint32_t)(key >> 32);
  const int sh = bits > 1 ? bits / 2 : 1;
  do {
    x = (x * 0x9E3779B1u) & mask;  x ^= x >> sh;  x = (x + k0) & mask;
    x = (x * 0x85EBCA6Bu) & mask;  x ^= x >> sh;  x = (x + k1) & mask;
    x = (x * 0xC2B2AE35u) & mask;  x ^= x >> sh;  x = (x + (k0 ^ (k1 * 0x27D4EB2Fu))) & mask;
    x = (x * 0x165667B1u) & mask;  x ^= x >> sh;
  } while (x >= N);
  return x;
}
// key_img[b]: the index that keys big image b's bijection -- its image index in the set it belongs to, so that a set
// matched inside a pooled call draws the subsets of its call alone
__global__ void k_subset_rows(const int64_t* __restrict__ img_off, const int32_t* __restrict__ big_img,
                              const int32_t* __restrict__ key_img, int64_t subset, uint64_t seed,
                              int32_t* __restrict__ vsrc, int32_t* __restrict__ vmap) {
  const int b = blockIdx.y, j = big_img[b];
  const uint32_t N = (uint32_t)(img_off[j + 1] - img_off[j]);
  const uint64_t key = seed * 0x9E3779B97F4A7C15ull + (uint64_t)(key_img[b] + 1) * 0xD1B54A32D192ED03ull;
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < subset; r += (int64_t)gridDim.x * blockDim.x) {
    const uint32_t loc = perm_in_range((uint32_t)r, N, key);
    vmap[b * subset + r] = (int32_t)loc;
    vsrc[b * subset + r] = (int32_t)(img_off[j] + loc);
  }
}
__global__ void k_gather_f32_rows(const float* __restrict__ src, const int32_t* __restrict__ rows, int64_t nrows, int D,
                                  float* __restrict__ dst) {
  const int64_t total = nrows * D;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / D;
    dst[i] = src[(int64_t)rows[r] * D + (i - r * D)];
  }
}
__global__ void k_gather_u16_rows(const uint4* __restrict__ src, const int32_t* __restrict__ rows, int64_t nrows, int chunks,
                                  uint4* __restrict__ dst) {
  const int64_t total = nrows * chunks;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / chunks;
    dst[i] = src[(int64_t)rows[r] * chunks + (i - r * chunks)];
  }
}

}  // namespace

int aps_k_subset_rows(cudaStream_t s, const int64_t* d_img_off, const int32_t* d_big_img, const int32_t* d_key_img,
                      int nbig, int64_t subset, uint64_t seed, int32_t* vsrc, int32_t* vmap) {
  if (nbig == 0 || subset == 0) return APS_OK;
  dim3 grid((unsigned)aps_min64(aps_ceil_div(subset, 256), 64), (unsigned)nbig);
  k_subset_rows<<<grid, 256, 0, s>>>(d_img_off, d_big_img, d_key_img, subset, seed, vsrc, vmap);
  APS_LAUNCHED();
  return APS_OK;
}
int aps_k_gather_f32_rows(cudaStream_t s, const float* src, const int32_t* rows, int64_t nrows, int D, float* dst) {
  if (nrows == 0) return APS_OK;
  k_gather_f32_rows<<<(unsigned)aps_min64(aps_ceil_div(nrows * D, 256), 148 * 16), 256, 0, s>>>(src, rows, nrows, D, dst);
  APS_LAUNCHED();
  return APS_OK;
}
int aps_k_gather_u16_rows(cudaStream_t s, const uint16_t* src, const int32_t* rows, int64_t nrows, int Dp, uint16_t* dst) {
  if (nrows == 0) return APS_OK;
  const int chunks = Dp * 2 / 16;
  k_gather_u16_rows<<<(unsigned)aps_min64(aps_ceil_div(nrows * chunks, 256), 148 * 16), 256, 0, s>>>(
      (const uint4*)src, rows, nrows, chunks, (uint4*)dst);
  APS_LAUNCHED();
  return APS_OK;
}

int aps_k_prepare_operands_f16(cudaStream_t s, const float* src, int64_t F, int D, int Dp, void* xh) {
  if (F == 0) return APS_OK;
  const unsigned grid = (unsigned)aps_min64(aps_ceil_div(F * (Dp / 8), 256), 148 * 16);
  k_prepare_operands_f16<<<grid, 256, 0, s>>>(src, F, D, Dp, (__half*)xh);
  APS_LAUNCHED();
  return APS_OK;
}

int aps_k_fill_f32(cudaStream_t s, float* dst, int64_t n, float v) {
  if (n <= 0) return APS_OK;
  k_fill_f32<<<(unsigned)aps_min64(aps_ceil_div(n, 256), 148 * 8), 256, 0, s>>>(dst, n, v);
  APS_LAUNCHED();
  return APS_OK;
}

int aps_k_image_sq_bounds(cudaStream_t s, const float* sq, const int64_t* d_start, const int64_t* d_count, int n, float2* out) {
  if (n == 0) return APS_OK;
  k_image_sq_bounds<<<n, 256, 0, s>>>(sq, d_start, d_count, out);
  APS_LAUNCHED();
  return APS_OK;
}

int aps_k_pair_screen(cudaStream_t s, int sm_count, const void* xh_q, int64_t Fq, const void* xh_t, int64_t Ft, int Dp,
                      const aps_pair_screen_tables& t, aps_tc_unit* d_units, int64_t n_units, uint32_t* out,
                      uint32_t* dump, int dump_tiles) {
  if (Dp != 64 && Dp != 128) {
    aps_set_error(APS_ERR_DIM, "", "pair screen supports padded descriptor lengths 64 and 128 (got %d)", Dp);
    return APS_ERR_DIM;
  }
  if (n_units <= 0 || t.npairs <= 0) return APS_OK;
  k_make_units<<<t.npairs, 32, 0, s>>>(t.qoff, t.qcnt, t.toff, t.tcnt, t.eoff, t.uoff, t.npairs, d_units);
  APS_LAUNCHED();
  CUtensorMap map_q, map_t;
  APS_TRY(make_map(&map_q, xh_q, Fq, Dp, TM, CU_TENSOR_MAP_DATA_TYPE_FLOAT16));
  APS_TRY(make_map(&map_t, xh_t, Ft, Dp, TN, CU_TENSOR_MAP_DATA_TYPE_FLOAT16));
  SParams P;
  P.units = d_units;
  P.n_units = n_units;
  P.dp = Dp;
  P.b_stages = Dp == 64 ? 8 : 4;
  P.a_bufs = Dp == 64 ? 2 : 1;
  P.out = out;
  P.dump = dump;
  P.dump_tiles = dump_tiles;
  P.idesc = make_idesc_f16_f16acc(TM, TN);
  const size_t smem = 1024 + (size_t)P.a_bufs * RB * TM * Dp * 2 + (size_t)P.b_stages * TN * Dp * 2 + sizeof(Bars);
  APS_CUDA(cudaFuncSetAttribute(k_pair_screen, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const unsigned grid = (unsigned)(n_units < sm_count ? n_units : sm_count);
  k_pair_screen<<<grid, NUM_THREADS, smem, s>>>(map_q, map_t, P);
  APS_LAUNCHED();
  return APS_OK;
}

int aps_k_pair_screen_decide(cudaStream_t s, const uint32_t* scr, const float* sq, const aps_pair_screen_tables& t,
                             const float2* img_bounds, const int32_t* flags, int Dp, double r2, double mt,
                             int32_t* survivors) {
  if (t.npairs <= 0) return APS_OK;
  APS_CUDA(cudaMemsetAsync(survivors, 0, (size_t)t.npairs * sizeof(int32_t), s));
  k_pair_screen_decide<<<t.npairs, 256, 0, s>>>(scr, sq, t.qoff, t.qcnt, t.timg, t.eoff, img_bounds, flags, Dp, r2, mt,
                                                survivors);
  APS_LAUNCHED();
  return APS_OK;
}
