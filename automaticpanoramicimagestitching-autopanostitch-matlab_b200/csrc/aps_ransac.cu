// aps_ransac.cu -- the consumer of the match lists (SURVEY.md section 8(f) rank 1): batched RANSAC homographies
// for the candidate image pairs, replacing the parfor of
//     PP/imageMatching/imageMatching.m:121-156            (pair loop, ni > 8 + 0.3 nf, inv(model))
//     PP/imageMatching/estimateTransformationRANSAC.m     :94-183 loop + refit, :188-225 normalised DLT,
//                                                         :444-516 findInliers, :518-530 checkModel,
//                                                         :532-572 isDegenerate, :574-596 normalizePoints
// ('projective', the only motion model PP/inputs.m:73 offers).  Double precision on CUDA cores.
//
// The reference loop is sequential only through its bookkeeping (best model so far, adaptive trial bound);
// given the minimal samples, every trial is independent.  So:
//   K-R1 k_ransac_samples : counter-based generator of n_draws x 4 distinct indices per pair (randperm stand-in)
//   K-R2a k_ransac_models : one THREAD per (pair, draw): normalised DLT of the 4 correspondences (A'A, cyclic
//                           Jacobi) and checkModel -> table of candidate models.
//   K-R2b k_ransac_eval   : one WARP per (pair, draw): lanes stride over the pair's correspondences (symmetric
//                           transfer error, consensus count, error sum, degeneracy of the consensus set;
//                           lane partial sums combined by a fixed butterfly).  Every operation is an explicit
//                           round-to-nearest intrinsic in the oracle's order, so (count, mean error) per draw
//                           carry the oracle's bits.  Draws are evaluated in waves [0,64) [64,256) [256,n):
//                           a pair whose loop has ended (adaptive bound) takes no part in later waves.
//   K-R3 k_ransac_scan    : one thread per pair replays the reference's bookkeeping over the per-draw results:
//                           trial / skipTrials counters, best = (more inliers, then smaller mean error),
//                           maxTrials = min(maxTrials, ceil(log(1-conf)/log(1-ratio^4))).
//   K-R4 k_ransac_final   : one CTA per pair: inlier mask of the best model, refit on all inliers
//                           (block-wide reductions for the centroids and A'A, Jacobi on one thread),
//                           checkModel + findInliers of the refit, acceptance rule, inverse.
// Work per draw ~ 250 double operations per correspondence; bound = FP64 pipe.  Data: 32 B per
// correspondence read by every thread of a pair at the same time (broadcast from L1).
#include <math_constants.h>

#include "aps_common.cuh"

#ifndef APS_FAIL
#define APS_FAIL(code, id, ...)           \
  do {                                    \
    aps_set_error(code, id, __VA_ARGS__); \
    return code;                          \
  } while (0)
#endif

namespace {

#define MUL(a, b) __dmul_rn((a), (b))
#define ADD(a, b) __dadd_rn((a), (b))
#define SUB(a, b) __dsub_rn((a), (b))
#define DIV(a, b) __ddiv_rn((a), (b))
#define SQRT(a) __dsqrt_rn((a))
constexpr double EPS64 = 2.220446049250313e-16;

// cyclic Jacobi, identical control flow to the oracle's (classical small-element rule, 50 sweeps max)
__device__ void jacobi9(double (*a)[9], double (*v)[9], double* d) {
  double b[9], z[9];
  for (int i = 0; i < 9; ++i) {
    for (int j = 0; j < 9; ++j) v[i][j] = (i == j) ? 1.0 : 0.0;
    b[i] = d[i] = a[i][i];
    z[i] = 0.0;
  }
  for (int sweep = 0; sweep < 50; ++sweep) {
    double sm = 0.0;
    for (int p = 0; p < 8; ++p)
      for (int q = p + 1; q < 9; ++q) sm = ADD(sm, fabs(a[p][q]));
    if (sm == 0.0) return;
    const double tresh = (sweep < 3) ? DIV(MUL(0.2, sm), 81.0) : 0.0;
    for (int p = 0; p < 8; ++p)
      for (int q = p + 1; q < 9; ++q) {
        const double apq = a[p][q];
        const double g = MUL(100.0, fabs(apq));
        if (sweep > 3 && ADD(fabs(d[p]), g) == fabs(d[p]) && ADD(fabs(d[q]), g) == fabs(d[q])) {
          a[p][q] = 0.0;
        } else if (fabs(apq) > tresh) {
          const double h = SUB(d[q], d[p]);
          double t;
          if (ADD(fabs(h), g) == fabs(h)) {
            t = DIV(apq, h);
          } else {
            const double theta = DIV(MUL(0.5, h), apq);
            t = DIV(1.0, ADD(fabs(theta), SQRT(ADD(1.0, MUL(theta, theta)))));
            if (theta < 0.0) t = -t;
          }
          const double c = DIV(1.0, SQRT(ADD(1.0, MUL(t, t))));
          const double s = MUL(t, c), tau = DIV(s, ADD(1.0, c)), hh = MUL(t, apq);
          z[p] = SUB(z[p], hh); z[q] = ADD(z[q], hh); d[p] = SUB(d[p], hh); d[q] = ADD(d[q], hh);
          a[p][q] = 0.0;
#define APS_ROT(M, i, j, k, l)                              \
  {                                                         \
    const double g_ = M[i][j], h_ = M[k][l];                \
    M[i][j] = SUB(g_, MUL(s, ADD(h_, MUL(g_, tau))));       \
    M[k][l] = ADD(h_, MUL(s, SUB(g_, MUL(h_, tau))));       \
  }
          for (int j = 0; j < p; ++j) APS_ROT(a, j, p, j, q)
          for (int j = p + 1; j < q; ++j) APS_ROT(a, p, j, j, q)
          for (int j = q + 1; j < 9; ++j) APS_ROT(a, p, j, q, j)
          for (int j = 0; j < 9; ++j) APS_ROT(v, j, p, j, q)
#undef APS_ROT
        }
      }
    for (int i = 0; i < 9; ++i) {
      b[i] = ADD(b[i], z[i]);
      d[i] = b[i];
      z[i] = 0.0;
    }
  }
}

// adds the two DLT rows of one normalised correspondence to the upper triangle of A'A
__device__ __forceinline__ void dlt_rows(double x, double y, double u, double v, double* r1, double* r2) {
  r1[0] = -x; r1[1] = -y; r1[2] = -1.0; r1[3] = 0.0; r1[4] = 0.0; r1[5] = 0.0; r1[6] = MUL(x, u); r1[7] = MUL(y, u); r1[8] = u;
  r2[0] = 0.0; r2[1] = 0.0; r2[2] = 0.0; r2[3] = -x; r2[4] = -y; r2[5] = -1.0; r2[6] = MUL(x, v); r2[7] = MUL(y, v); r2[8] = v;
}

// H = T2 \ (Hn / Hn(3,3)) * T1 from the eigenvector of the smallest eigenvalue of M = A'A
__device__ void homography_from_gram(double (*M)[9], const double* T1, const double* T2, double* H) {
  double V[9][9], d[9];
  jacobi9(M, V, d);
  int im = 0;
  for (int i = 1; i < 9; ++i)
    if (d[i] < d[im]) im = i;
  double Hn[9], X[9];
  const double h33 = V[8][im];
  for (int i = 0; i < 9; ++i) Hn[i] = DIV(V[i][im], h33);
  for (int j = 0; j < 3; ++j) {
    X[6 + j] = Hn[6 + j];
    X[j] = DIV(SUB(Hn[j], MUL(T2[1], Hn[6 + j])), T2[0]);
    X[3 + j] = DIV(SUB(Hn[3 + j], MUL(T2[2], Hn[6 + j])), T2[0]);
  }
  for (int i = 0; i < 3; ++i) {
    H[3 * i + 0] = MUL(X[3 * i + 0], T1[0]);
    H[3 * i + 1] = MUL(X[3 * i + 1], T1[0]);
    H[3 * i + 2] = ADD(ADD(MUL(X[3 * i + 0], T1[1]), MUL(X[3 * i + 1], T1[2])), X[3 * i + 2]);
  }
}

// normalizePoints of four correspondences (sequential sums in index order)
__device__ void normalize4(const double2* p, const uint32_t* s, double* T) {
  double sx = 0.0, sy = 0.0;
  for (int i = 0; i < 4; ++i) {
    sx = ADD(sx, p[s[i]].x);
    sy = ADD(sy, p[s[i]].y);
  }
  const double cx = DIV(sx, 4.0), cy = DIV(sy, 4.0);
  double sd = 0.0;
  for (int i = 0; i < 4; ++i) {
    const double dx = SUB(p[s[i]].x, cx), dy = SUB(p[s[i]].y, cy);
    sd = ADD(sd, SQRT(ADD(MUL(dx, dx), MUL(dy, dy))));
  }
  const double scale = DIV(1.0, DIV(sd, 4.0));
  T[0] = scale;
  T[1] = MUL(-scale, cx);
  T[2] = MUL(-scale, cy);
}

__device__ void homography4(const double2* p1, const double2* p2, const uint32_t* s, double* H) {
  double T1[3], T2[3], M[9][9];
  normalize4(p1, s, T1);
  normalize4(p2, s, T2);
  for (int a = 0; a < 9; ++a)
    for (int b = 0; b < 9; ++b) M[a][b] = 0.0;
  for (int i = 0; i < 4; ++i) {
    const double x = ADD(MUL(T1[0], p1[s[i]].x), T1[1]), y = ADD(MUL(T1[0], p1[s[i]].y), T1[2]);
    const double u = ADD(MUL(T2[0], p2[s[i]].x), T2[1]), v = ADD(MUL(T2[0], p2[s[i]].y), T2[2]);
    double r1[9], r2[9];
    dlt_rows(x, y, u, v, r1, r2);
    for (int a = 0; a < 9; ++a)
      for (int b = a; b < 9; ++b) M[a][b] = ADD(M[a][b], ADD(MUL(r1[a], r1[b]), MUL(r2[a], r2[b])));
  }
  homography_from_gram(M, T1, T2, H);
}

__device__ __forceinline__ double det3(const double* H) {
  return ADD(SUB(MUL(H[0], SUB(MUL(H[4], H[8]), MUL(H[5], H[7]))), MUL(H[1], SUB(MUL(H[3], H[8]), MUL(H[5], H[6])))),
             MUL(H[2], SUB(MUL(H[3], H[7]), MUL(H[4], H[6]))));
}
__device__ __forceinline__ void adj3(const double* H, double* A) {
  A[0] = SUB(MUL(H[4], H[8]), MUL(H[5], H[7])); A[1] = SUB(MUL(H[2], H[7]), MUL(H[1], H[8])); A[2] = SUB(MUL(H[1], H[5]), MUL(H[2], H[4]));
  A[3] = SUB(MUL(H[5], H[6]), MUL(H[3], H[8])); A[4] = SUB(MUL(H[0], H[8]), MUL(H[2], H[6])); A[5] = SUB(MUL(H[2], H[3]), MUL(H[0], H[5]));
  A[6] = SUB(MUL(H[3], H[7]), MUL(H[4], H[6])); A[7] = SUB(MUL(H[1], H[6]), MUL(H[0], H[7])); A[8] = SUB(MUL(H[0], H[4]), MUL(H[1], H[3]));
}
__device__ __forceinline__ double norm1_3(const double* H) {
  double m = 0.0;
  for (int j = 0; j < 3; ++j) {
    const double c = ADD(ADD(fabs(H[j]), fabs(H[3 + j])), fabs(H[6 + j]));
    if (c > m) m = c;
  }
  return m;
}
// checkModel: finite, |det| > eps, exact 1-norm rcond > eps
__device__ bool check_model(const double* H) {
  for (int i = 0; i < 9; ++i)
    if (!isfinite(H[i])) return false;
  const double det = det3(H);
  if (!(fabs(det) > EPS64)) return false;
  double A[9];
  adj3(H, A);
  for (int i = 0; i < 9; ++i) A[i] = DIV(A[i], det);
  return DIV(1.0, MUL(norm1_3(H), norm1_3(A))) > EPS64;
}

struct LU3 {
  double L10, L20, L21, U0, U1, U2, U3, U4, U5;
  int p0, p1, p2;
};
__device__ void lu3(const double* H, LU3& f) {
  double a[3][3] = {{H[0], H[1], H[2]}, {H[3], H[4], H[5]}, {H[6], H[7], H[8]}};
  int pv[3] = {0, 1, 2};
  int m = 0;
  if (fabs(a[1][0]) > fabs(a[m][0])) m = 1;
  if (fabs(a[2][0]) > fabs(a[m][0])) m = 2;
  if (m != 0) {
    for (int j = 0; j < 3; ++j) { const double t = a[0][j]; a[0][j] = a[m][j]; a[m][j] = t; }
    const int t = pv[0]; pv[0] = pv[m]; pv[m] = t;
  }
  a[1][0] = DIV(a[1][0], a[0][0]);
  a[2][0] = DIV(a[2][0], a[0][0]);
  a[1][1] = SUB(a[1][1], MUL(a[1][0], a[0][1])); a[1][2] = SUB(a[1][2], MUL(a[1][0], a[0][2]));
  a[2][1] = SUB(a[2][1], MUL(a[2][0], a[0][1])); a[2][2] = SUB(a[2][2], MUL(a[2][0], a[0][2]));
  if (fabs(a[2][1]) > fabs(a[1][1])) {
    for (int j = 0; j < 3; ++j) { const double t = a[1][j]; a[1][j] = a[2][j]; a[2][j] = t; }
    const int t = pv[1]; pv[1] = pv[2]; pv[2] = t;
  }
  a[2][1] = DIV(a[2][1], a[1][1]);
  a[2][2] = SUB(a[2][2], MUL(a[2][1], a[1][2]));
  f.L10 = a[1][0]; f.L20 = a[2][0]; f.L21 = a[2][1];
  f.U0 = a[0][0]; f.U1 = a[0][1]; f.U2 = a[0][2]; f.U3 = a[1][1]; f.U4 = a[1][2]; f.U5 = a[2][2];
  f.p0 = pv[0]; f.p1 = pv[1]; f.p2 = pv[2];
}

// symmetric transfer error of one correspondence ((x,y) -> (u,v)) under H
__device__ __forceinline__ double point_error(const double* H, const LU3& f, double x, double y, double u, double v) {
  const double t2 = ADD(ADD(MUL(H[6], x), MUL(H[7], y)), H[8]);
  const double tx = DIV(ADD(ADD(MUL(H[0], x), MUL(H[1], y)), H[2]), t2);
  const double ty = DIV(ADD(ADD(MUL(H[3], x), MUL(H[4], y)), H[5]), t2);
  const double b0 = (f.p0 == 0) ? u : (f.p0 == 1 ? v : 1.0);
  const double b1 = (f.p1 == 0) ? u : (f.p1 == 1 ? v : 1.0);
  const double b2 = (f.p2 == 0) ? u : (f.p2 == 1 ? v : 1.0);
  const double y0 = b0;
  const double y1 = SUB(b1, MUL(f.L10, y0));
  const double y2 = SUB(SUB(b2, MUL(f.L20, y0)), MUL(f.L21, y1));
  const double w2 = DIV(y2, f.U5);
  const double w1 = DIV(SUB(y1, MUL(f.U4, w2)), f.U3);
  const double w0 = DIV(SUB(SUB(y0, MUL(f.U1, w1)), MUL(f.U2, w2)), f.U0);
  const double ix = DIV(w0, w2), iy = DIV(w1, w2);
  const double ex = SUB(u, tx), ey = SUB(v, ty), fx = SUB(x, ix), fy = SUB(y, iy);
  const double d1 = ADD(MUL(ex, ex), MUL(ey, ey));
  const double d2 = ADD(MUL(fx, fx), MUL(fy, fy));
  double e = SQRT(ADD(d1, d2));
  if (!isfinite(e)) e = CUDART_INF;
  if (!isfinite(DIV(t2, t2))) e = CUDART_INF;
  return e;
}

__device__ __forceinline__ bool degenerate_ratio(double sxx, double sxy, double syy) {
  const double hd = MUL(0.5, SUB(sxx, syy));
  const double l1 = ADD(MUL(0.5, ADD(sxx, syy)), SQRT(ADD(MUL(hd, hd), MUL(sxy, sxy))));
  const double l2 = DIV(SUB(MUL(sxx, syy), MUL(sxy, sxy)), l1);
  const double ratio = DIV(SQRT(fmax(l2, 0.0)), SQRT(l1));
  return ratio < 1e-3;
}

__device__ __forceinline__ uint64_t splitmix64(uint64_t& s) {
  uint64_t z = (s += 0x9E3779B97F4A7C15ull);
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

// K-R1: four distinct indices per (pair, draw), uniform without replacement (stand-in for randperm(n, 4)).  The draws
// of pair p are keyed by keys[p] (its index in its own set's candidate list), or by p when keys is NULL.
__global__ void k_ransac_samples(const int64_t* __restrict__ pt_ptr, const int64_t* __restrict__ keys, int64_t n_draws,
                                 uint64_t seed, uint32_t* __restrict__ samples) {
  const int64_t pair = blockIdx.y;
  const int64_t key = keys ? keys[pair] : pair;
  const int64_t d = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= n_draws) return;
  const int64_t n = pt_ptr[pair + 1] - pt_ptr[pair];
  uint32_t* out = samples + (pair * n_draws + d) * 4;
  if (n < 4) {
    out[0] = out[1] = out[2] = out[3] = 0;
    return;
  }
  uint64_t s = seed ^ (0xD1B54A32D192ED03ull * (uint64_t)(key + 1)) ^ (0x8CB92BA72F3D8DD7ull * (uint64_t)(d + 1));
  uint32_t c[4];
  for (int k = 0; k < 4; ++k) {
    uint32_t r = (uint32_t)(splitmix64(s) % (uint64_t)(n - k));
    // map r to the r-th index not chosen yet: walk the chosen ones in ascending order
    uint32_t srt[4];
    for (int i = 0; i < k; ++i) srt[i] = c[i];
    for (int i = 1; i < k; ++i)
      for (int j = i; j > 0 && srt[j] < srt[j - 1]; --j) { const uint32_t t = srt[j]; srt[j] = srt[j - 1]; srt[j - 1] = t; }
    for (int i = 0; i < k; ++i)
      if (r >= srt[i]) ++r;
    c[k] = r;
  }
  out[0] = c[0]; out[1] = c[1]; out[2] = c[2]; out[3] = c[3];
}

// K-R2a: one thread per (pair, draw): normalised DLT of the four sampled correspondences + checkModel.
// Hs[slot] = the 3x3 model (row-major); cnt_out[slot] = -1 marks a skipped sample.
__global__ void __launch_bounds__(128) k_ransac_models(const int64_t* __restrict__ pt_ptr, const double2* __restrict__ p1,
                                                       const double2* __restrict__ p2, const uint32_t* __restrict__ samples,
                                                       int64_t n_draws, int64_t d0, int64_t d1,
                                                       const uint8_t* __restrict__ done, double* __restrict__ Hs,
                                                       int32_t* __restrict__ cnt_out, double* __restrict__ err_out) {
  const int64_t pair = blockIdx.y;
  const int64_t d = d0 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= d1 || done[pair]) return;  // the pair's loop already ended inside an earlier wave of draws
  const int64_t o = pt_ptr[pair], n = pt_ptr[pair + 1] - o;
  const int64_t slot = pair * n_draws + d;
  cnt_out[slot] = -1;
  err_out[slot] = CUDART_INF;
  if (n < 4) return;
  uint32_t s[4];
  for (int i = 0; i < 4; ++i) s[i] = samples[slot * 4 + i];
  for (int i = 0; i < 4; ++i)
    if ((int64_t)s[i] >= n) return;  // caller-supplied table with an index outside the pair: a skipped sample
  double H[9];
  homography4(p1 + o, p2 + o, s, H);
  if (!check_model(H)) return;
  for (int i = 0; i < 9; ++i) Hs[slot * 9 + i] = H[i];
  cnt_out[slot] = 0;
}

// butterfly total of the lanes' partial sums (offsets 16, 8, 4, 2, 1): every lane ends with the same bits
__device__ __forceinline__ double warp_total(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = ADD(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// K-R2b: one WARP per (pair, draw): lanes stride over the pair's correspondences (point r -> lane r mod 32),
// symmetric transfer error, consensus count, error sum and the degeneracy test of the consensus set.
// cnt_out = size of the consensus set (0 when degenerate), err_out = its mean error (cnt >= 4).
__global__ void __launch_bounds__(128) k_ransac_eval(const int64_t* __restrict__ pt_ptr, const double2* __restrict__ p1,
                                                     const double2* __restrict__ p2, int64_t n_draws, int64_t d0,
                                                     int64_t d1, const uint8_t* __restrict__ done,
                                                     const double* __restrict__ Hs, double thr,
                                                     int32_t* __restrict__ cnt_out, double* __restrict__ err_out) {
  const int64_t pair = blockIdx.y;
  const int lane = threadIdx.x & 31;
  const int64_t d = d0 + (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (d >= d1 || done[pair]) return;
  const int64_t slot = pair * n_draws + d;
  if (cnt_out[slot] < 0) return;  // skipped sample (warp-uniform)
  const int64_t o = pt_ptr[pair], n = pt_ptr[pair + 1] - o;
  const double2* q1 = p1 + o;
  const double2* q2 = p2 + o;
  double H[9];
  for (int i = 0; i < 9; ++i) H[i] = Hs[slot * 9 + i];
  LU3 f;
  lu3(H, f);
  int32_t c = 0;
  double es = 0.0, sx = 0.0, sy = 0.0;
  for (int64_t r = lane; r < n; r += 32) {
    const double2 a = q1[r], b = q2[r];
    const double e = point_error(H, f, a.x, a.y, b.x, b.y);
    if (e < thr) {
      ++c;
      es = ADD(es, e);
      sx = ADD(sx, a.x);
      sy = ADD(sy, a.y);
    }
  }
  int32_t cnt = __reduce_add_sync(0xffffffffu, c);
  es = warp_total(es);
  if (cnt >= 4) {
    const double mx = DIV(warp_total(sx), (double)cnt), my = DIV(warp_total(sy), (double)cnt);
    double sxx = 0.0, sxy = 0.0, syy = 0.0;
    for (int64_t r = lane; r < n; r += 32) {
      const double2 a = q1[r], b = q2[r];
      const double e = point_error(H, f, a.x, a.y, b.x, b.y);
      if (e < thr) {
        const double dx = SUB(a.x, mx), dy = SUB(a.y, my);
        sxx = ADD(sxx, MUL(dx, dx));
        sxy = ADD(sxy, MUL(dx, dy));
        syy = ADD(syy, MUL(dy, dy));
      }
    }
    if (degenerate_ratio(warp_total(sxx), warp_total(sxy), warp_total(syy))) cnt = 0;
  }
  if (lane == 0) {
    cnt_out[slot] = cnt;
    err_out[slot] = (cnt >= 4) ? DIV(es, (double)cnt) : CUDART_INF;
  }
}

// K-R3: the reference's sequential bookkeeping over the per-draw results
__global__ void k_ransac_scan(int64_t n_pairs, const int64_t* __restrict__ pt_ptr, const int32_t* __restrict__ cnt,
                              const double* __restrict__ err, int64_t n_draws, int64_t d_limit, double confidence,
                              int max_trials_in, int32_t* __restrict__ best_draw, int32_t* __restrict__ draws_used,
                              uint8_t* __restrict__ done) {
  const int64_t pair = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (pair >= n_pairs) return;
  if (done[pair]) return;  // finished in an earlier wave: results stand
  const int64_t n = pt_ptr[pair + 1] - pt_ptr[pair];
  int32_t best = -1, bestCnt = 0;
  double bestErr = CUDART_INF;
  int64_t d = 0;
  if (n >= 4) {
    double maxTrials = (double)max_trials_in;
    const int64_t maxSkip = (int64_t)max_trials_in * 10;
    int64_t trial = 1, skip = 0;
    const double lc = log(SUB(1.0, DIV(confidence, 100.0)));
    while ((double)trial <= maxTrials && skip < maxSkip && d < d_limit) {
      const int32_t c = cnt[pair * n_draws + d];
      const double e = err[pair * n_draws + d];
      const int32_t dd = (int32_t)d;
      ++d;
      if (c < 0) {
        ++skip;
        continue;
      }
      if (c >= 4 && (c > bestCnt || (c == bestCnt && e < bestErr))) {
        best = dd;
        bestCnt = c;
        bestErr = e;
        const double ratio = DIV((double)c, (double)n);
        if (ratio > 0.0) {
          const double r2 = MUL(ratio, ratio);
          const double t = ceil(DIV(lc, log(SUB(1.0, MUL(r2, r2)))));
          if (t < maxTrials) maxTrials = t;
        }
      }
      ++trial;
    }
    // the reference's loop ended by its own conditions (not because this wave of draws ran out)
    done[pair] = !((double)trial <= maxTrials && skip < maxSkip) || d_limit >= n_draws;
  } else {
    done[pair] = 1;
  }
  best_draw[pair] = best;
  draws_used[pair] = (int32_t)d;
}

__device__ __forceinline__ double block_sum(double v, double* red) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31, nw = blockDim.x >> 5;
  __syncthreads();
  if (l == 0) red[w] = v;
  __syncthreads();
  double t = 0.0;
  for (int i = 0; i < nw; ++i) t += red[i];  // same order in every thread: all threads hold the same sum
  return t;
}

// K-R4: one CTA per pair: refit on the consensus set of the best draw and the reference's final decisions
__global__ void __launch_bounds__(256) k_ransac_final(const int64_t* __restrict__ pt_ptr, const double2* __restrict__ p1,
                                                      const double2* __restrict__ p2, const double* __restrict__ Hs_tab,
                                                      int64_t n_draws, double thr, const int32_t* __restrict__ best_draw,
                                                      uint8_t* __restrict__ mask_best, double* __restrict__ models,
                                                      double* __restrict__ models_inv, uint8_t* __restrict__ inliers,
                                                      int32_t* __restrict__ n_inliers, uint8_t* __restrict__ accepted) {
  __shared__ double red[8];
  __shared__ double Hs[9], Hr[9];
  __shared__ double Ms[45];
  __shared__ int flag;
  const int64_t pair = blockIdx.x;
  const int64_t o = pt_ptr[pair], n = pt_ptr[pair + 1] - o;
  const double2* q1 = p1 + o;
  const double2* q2 = p2 + o;
  const int tid = threadIdx.x;
  const int bd = best_draw[pair];
  const double qnan = __longlong_as_double(0x7ff8000000000000ll);
  if (bd < 0) {  // nothing found (or nf < 4): model = [], no inliers
    for (int64_t r = tid; r < n; r += blockDim.x) inliers[o + r] = 0;
    if (tid < 9) { models[pair * 9 + tid] = qnan; models_inv[pair * 9 + tid] = qnan; }
    if (tid == 0) { n_inliers[pair] = 0; accepted[pair] = 0; }
    return;
  }
  if (tid < 9) Hs[tid] = Hs_tab[(pair * n_draws + bd) * 9 + tid];
  __syncthreads();
  double H[9];
  for (int i = 0; i < 9; ++i) H[i] = Hs[i];
  LU3 f;
  lu3(H, f);
  // consensus set of the best draw (known non-degenerate: K-R2 decided that with the oracle's bits)
  double c0 = 0.0, s1x = 0.0, s1y = 0.0, s2x = 0.0, s2y = 0.0;
  for (int64_t r = tid; r < n; r += blockDim.x) {
    const double2 a = q1[r], b = q2[r];
    const bool in = point_error(H, f, a.x, a.y, b.x, b.y) < thr;
    mask_best[o + r] = (uint8_t)in;
    if (in) { c0 += 1.0; s1x += a.x; s1y += a.y; s2x += b.x; s2y += b.y; }
  }
  const double cntb = block_sum(c0, red);
  const double m1x = block_sum(s1x, red) / cntb, m1y = block_sum(s1y, red) / cntb;
  const double m2x = block_sum(s2x, red) / cntb, m2y = block_sum(s2y, red) / cntb;
  double sd1 = 0.0, sd2 = 0.0;
  for (int64_t r = tid; r < n; r += blockDim.x)
    if (mask_best[o + r]) {
      const double2 a = q1[r], b = q2[r];
      sd1 += sqrt((a.x - m1x) * (a.x - m1x) + (a.y - m1y) * (a.y - m1y));
      sd2 += sqrt((b.x - m2x) * (b.x - m2x) + (b.y - m2y) * (b.y - m2y));
    }
  double T1[3], T2[3];
  T1[0] = 1.0 / (block_sum(sd1, red) / cntb); T1[1] = -T1[0] * m1x; T1[2] = -T1[0] * m1y;
  T2[0] = 1.0 / (block_sum(sd2, red) / cntb); T2[1] = -T2[0] * m2x; T2[2] = -T2[0] * m2y;
  // A'A over the consensus set: per-thread partial upper triangles, then 45 block reductions
  double acc[45];
#pragma unroll
  for (int i = 0; i < 45; ++i) acc[i] = 0.0;
  for (int64_t r = tid; r < n; r += blockDim.x)
    if (mask_best[o + r]) {
      const double2 a = q1[r], b = q2[r];
      const double x = T1[0] * a.x + T1[1], y = T1[0] * a.y + T1[2];
      const double u = T2[0] * b.x + T2[1], v = T2[0] * b.y + T2[2];
      double r1[9], r2[9];
      dlt_rows(x, y, u, v, r1, r2);
      int k = 0;
#pragma unroll
      for (int i = 0; i < 9; ++i)
#pragma unroll
        for (int j = i; j < 9; ++j) acc[k++] += r1[i] * r1[j] + r2[i] * r2[j];
    }
#pragma unroll
  for (int i = 0; i < 45; ++i) {
    const double t = block_sum(acc[i], red);
    if (tid == 0) Ms[i] = t;
  }
  __syncthreads();
  if (tid == 0) {
    double M[9][9];
    int k = 0;
    for (int i = 0; i < 9; ++i)
      for (int j = 0; j < 9; ++j) M[i][j] = 0.0;
    for (int i = 0; i < 9; ++i)
      for (int j = i; j < 9; ++j) M[i][j] = Ms[k++];
    double Hf[9];
    homography_from_gram(M, T1, T2, Hf);
    for (int i = 0; i < 9; ++i) Hr[i] = Hf[i];
    flag = check_model(Hf) ? 1 : 0;
  }
  __syncthreads();
  bool use_best = true;
  double cntr = 0.0;
  if (flag) {
    double G[9];
    for (int i = 0; i < 9; ++i) G[i] = Hr[i];
    LU3 g;
    lu3(G, g);
    double c1 = 0.0, sx = 0.0, sy = 0.0;
    for (int64_t r = tid; r < n; r += blockDim.x) {
      const double2 a = q1[r], b = q2[r];
      const bool in = point_error(G, g, a.x, a.y, b.x, b.y) < thr;
      inliers[o + r] = (uint8_t)in;
      if (in) { c1 += 1.0; sx += a.x; sy += a.y; }
    }
    cntr = block_sum(c1, red);
    if (cntr >= 4.0) {
      const double mx = block_sum(sx, red) / cntr, my = block_sum(sy, red) / cntr;
      double sxx = 0.0, sxy = 0.0, syy = 0.0;
      for (int64_t r = tid; r < n; r += blockDim.x)
        if (inliers[o + r]) {
          const double dx = q1[r].x - mx, dy = q1[r].y - my;
          sxx += dx * dx; sxy += dx * dy; syy += dy * dy;
        }
      sxx = block_sum(sxx, red); sxy = block_sum(sxy, red); syy = block_sum(syy, red);
      use_best = degenerate_ratio(sxx, sxy, syy);  // degenerate refit consensus -> 0 inliers -> keep the best draw
    }
  }
  if (use_best) {
    for (int64_t r = tid; r < n; r += blockDim.x) inliers[o + r] = mask_best[o + r];
    cntr = cntb;
  }
  if (tid == 0) {
    const double* Hm = use_best ? Hs : Hr;
    const int32_t ni = (int32_t)cntr;
    n_inliers[pair] = ni;
    const bool acc_ok = (double)ni > 8.0 + 0.3 * (double)n;  // imageMatching.m:147
    accepted[pair] = acc_ok ? 1 : 0;
    double A[9];
    adj3(Hm, A);
    const double det = det3(Hm);
    for (int i = 0; i < 9; ++i) {
      models[pair * 9 + i] = Hm[i];
      models_inv[pair * 9 + i] = acc_ok ? A[i] / det : qnan;
    }
  }
}

// hand-off from the matching stage (refineMatch, imageMatching.m:224-227): gathers the matched keypoints of the
// candidate pairs.  Correspondence i of pair p = match row (a, b), 1-based: p2 = keypoints{ii}(a,:), p1 = keypoints{jj}(b,:)
// (the reference calls estimateTransformationRANSAC(matchedPts_2, matchedPts_1, ...)).
__global__ void k_gather_matched_points(const int64_t* __restrict__ pt_ptr, const uint32_t* __restrict__ rows,
                                        const int32_t* __restrict__ pair_ii, const int32_t* __restrict__ pair_jj,
                                        const int64_t* __restrict__ img_off, const double2* __restrict__ kp,
                                        double2* __restrict__ p1, double2* __restrict__ p2) {
  const int64_t pair = blockIdx.y;
  const int64_t o = pt_ptr[pair], n = pt_ptr[pair + 1] - o;
  const int64_t oi = img_off[pair_ii[pair]], oj = img_off[pair_jj[pair]];
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (int64_t)gridDim.x * blockDim.x) {
    p2[o + r] = kp[oi + (int64_t)rows[2 * (o + r)] - 1];
    p1[o + r] = kp[oj + (int64_t)rows[2 * (o + r) + 1] - 1];
  }
}

}  // namespace

// ---- launchers ------------------------------------------------------------------------------------------------
static int ransac_device(aps_ctx* c, int64_t n_pairs, int64_t total, const int64_t* d_ptr, const double2* d_p1,
                         const double2* d_p2, uint32_t* d_samples, bool have_samples, const int64_t* d_keys,
                         int64_t n_draws, uint64_t seed, double max_distance, double confidence, int max_trials,
                         double* d_models, double* d_minv, uint8_t* d_inl, int32_t* d_ninl, uint8_t* d_acc,
                         int32_t* d_used) {
  cudaStream_t s = c->stream;
  const dim3 gd((unsigned)((n_draws + 127) / 128), (unsigned)n_pairs);
  if (!have_samples) {
    k_ransac_samples<<<gd, 128, 0, s>>>(d_ptr, d_keys, n_draws, seed, d_samples);
    APS_LAUNCHED();
  }
  DevBuf<int32_t> cnt, best;
  DevBuf<double> err, Htab;
  DevBuf<uint8_t> mask, done;
  APS_TRY(Htab.alloc((size_t)(n_pairs * n_draws) * 9, s));
  APS_TRY(done.alloc((size_t)n_pairs, s));
  APS_CUDA(cudaMemsetAsync(done.p, 0, (size_t)n_pairs, s));
  APS_TRY(cnt.alloc((size_t)(n_pairs * n_draws), s));
  APS_TRY(err.alloc((size_t)(n_pairs * n_draws), s));
  APS_TRY(best.alloc((size_t)n_pairs, s));
  APS_TRY(mask.alloc((size_t)(total > 0 ? total : 1), s));
  // Draws are evaluated in waves [0,64), [64,256), [256,n_draws): the adaptive trial bound ends most loops
  // within the first wave, and a pair whose loop has ended takes no part in later waves.  Every wave
  // replays the bookkeeping from draw 0, so the outcome is that of one sequential pass.
  const int64_t edges[4] = {0, 64, 256, n_draws};
  for (int w = 0; w < 3; ++w) {
    const int64_t d0 = edges[w] < n_draws ? edges[w] : n_draws, d1 = edges[w + 1] < n_draws ? edges[w + 1] : n_draws;
    if (d1 <= d0) continue;
    const dim3 gm((unsigned)((d1 - d0 + 127) / 128), (unsigned)n_pairs);
    k_ransac_models<<<gm, 128, 0, s>>>(d_ptr, d_p1, d_p2, d_samples, n_draws, d0, d1, done.p, Htab.p, cnt.p, err.p);
    APS_LAUNCHED();
    const dim3 ge((unsigned)((d1 - d0 + 3) / 4), (unsigned)n_pairs);
    k_ransac_eval<<<ge, 128, 0, s>>>(d_ptr, d_p1, d_p2, n_draws, d0, d1, done.p, Htab.p, max_distance, cnt.p, err.p);
    APS_LAUNCHED();
    k_ransac_scan<<<(unsigned)((n_pairs + 63) / 64), 64, 0, s>>>(n_pairs, d_ptr, cnt.p, err.p, n_draws, d1, confidence,
                                                                 max_trials, best.p, d_used, done.p);
    APS_LAUNCHED();
  }
  k_ransac_final<<<(unsigned)n_pairs, 256, 0, s>>>(d_ptr, d_p1, d_p2, Htab.p, n_draws, max_distance, best.p, mask.p,
                                                   d_models, d_minv, d_inl, d_ninl, d_acc);
  APS_LAUNCHED();
  return APS_OK;
}

static int ransac_params(int64_t n_draws, int max_trials, double confidence) {
  if (n_draws <= 0 || max_trials <= 0) APS_FAIL(APS_ERR_ARGS, "", "n_draws and max_trials must be positive");
  if (!(confidence > 0.0 && confidence < 100.0)) APS_FAIL(APS_ERR_ARGS, "", "confidence must be in (0, 100)");
  return APS_OK;
}

static int ransac_args(aps_ctx* c, int64_t n_pairs, const int64_t* pt_ptr, int64_t n_draws, int max_trials,
                       double confidence) {
  if (!c) APS_FAIL(APS_ERR_NOGPU, "apsmatch:nogpu", "context is NULL (no GPU context; there is no CPU path)");
  if (n_pairs < 0 || (n_pairs > 0 && !pt_ptr)) APS_FAIL(APS_ERR_ARGS, "", "bad pair list");
  APS_TRY(ransac_params(n_draws, max_trials, confidence));
  if (n_pairs > 65535) APS_FAIL(APS_ERR_ARGS, "", "at most 65535 candidate pairs per call");
  for (int64_t p = 0; p < n_pairs; ++p)
    if (pt_ptr[p + 1] < pt_ptr[p]) APS_FAIL(APS_ERR_ARGS, "", "pt_ptr must be non-decreasing");
  return APS_OK;
}

extern "C" int aps_ransac_sample_table(aps_ctx* c, const int64_t* pt_ptr, int64_t n_pairs, int64_t n_draws,
                                       uint64_t seed, uint32_t* samples) {
  APS_TRY(ransac_args(c, n_pairs, pt_ptr, n_draws, 1, 50.0));
  APS_CUDA(cudaSetDevice(c->device));
  if (n_pairs == 0) return APS_OK;
  if (!samples) APS_FAIL(APS_ERR_ARGS, "", "samples is NULL");
  DevBuf<int64_t> dptr;
  DevBuf<uint32_t> ds;
  APS_TRY(dptr.alloc((size_t)n_pairs + 1, c->stream));
  APS_TRY(ds.alloc((size_t)(n_pairs * n_draws * 4), c->stream));
  APS_CUDA(cudaMemcpyAsync(dptr.p, pt_ptr, (size_t)(n_pairs + 1) * 8, cudaMemcpyHostToDevice, c->stream));
  const dim3 gd((unsigned)((n_draws + 127) / 128), (unsigned)n_pairs);
  k_ransac_samples<<<gd, 128, 0, c->stream>>>(dptr.p, nullptr, n_draws, seed, ds.p);
  APS_LAUNCHED();
  APS_CUDA(cudaMemcpyAsync(samples, ds.p, (size_t)(n_pairs * n_draws * 4) * 4, cudaMemcpyDeviceToHost, c->stream));
  APS_CUDA(cudaStreamSynchronize(c->stream));
  return APS_OK;
}

extern "C" int aps_image_matching_batch(aps_ctx* c, int64_t n_pairs, const int64_t* pt_ptr, const double* pts1,
                                        const double* pts2, double max_distance, double confidence, int max_trials,
                                        const uint32_t* samples, int64_t n_draws, uint64_t seed, double* models,
                                        double* models_inv, uint8_t* inliers, int32_t* n_inliers, uint8_t* accepted,
                                        int32_t* draws_used) {
  APS_TRY(ransac_args(c, n_pairs, pt_ptr, n_draws, max_trials, confidence));
  APS_CUDA(cudaSetDevice(c->device));
  if (n_pairs == 0) return APS_OK;
  const int64_t base = pt_ptr[0], total = pt_ptr[n_pairs] - base;
  if (base != 0) APS_FAIL(APS_ERR_ARGS, "", "pt_ptr[0] must be 0");
  if ((total > 0 && (!pts1 || !pts2 || !inliers)) || !models || !models_inv || !n_inliers || !accepted || !draws_used)
    APS_FAIL(APS_ERR_ARGS, "", "NULL argument");
  cudaStream_t s = c->stream;
  DevBuf<int64_t> dptr;
  DevBuf<double2> dp1, dp2;
  DevBuf<uint32_t> ds;
  DevBuf<double> dm, dmi;
  DevBuf<uint8_t> dinl, dacc;
  DevBuf<int32_t> dni, dused;
  const size_t tot = (size_t)(total > 0 ? total : 1);
  APS_TRY(dptr.alloc((size_t)n_pairs + 1, s));
  APS_TRY(dp1.alloc(tot, s));
  APS_TRY(dp2.alloc(tot, s));
  APS_TRY(ds.alloc((size_t)(n_pairs * n_draws * 4), s));
  APS_TRY(dm.alloc((size_t)n_pairs * 9, s));
  APS_TRY(dmi.alloc((size_t)n_pairs * 9, s));
  APS_TRY(dinl.alloc(tot, s));
  APS_TRY(dacc.alloc((size_t)n_pairs, s));
  APS_TRY(dni.alloc((size_t)n_pairs, s));
  APS_TRY(dused.alloc((size_t)n_pairs, s));
  APS_CUDA(cudaMemcpyAsync(dptr.p, pt_ptr, (size_t)(n_pairs + 1) * 8, cudaMemcpyHostToDevice, s));
  if (total > 0) {
    APS_CUDA(cudaMemcpyAsync(dp1.p, pts1, (size_t)total * 16, cudaMemcpyHostToDevice, s));
    APS_CUDA(cudaMemcpyAsync(dp2.p, pts2, (size_t)total * 16, cudaMemcpyHostToDevice, s));
  }
  if (samples)
    APS_CUDA(cudaMemcpyAsync(ds.p, samples, (size_t)(n_pairs * n_draws * 4) * 4, cudaMemcpyHostToDevice, s));
  APS_TRY(ransac_device(c, n_pairs, total, dptr.p, dp1.p, dp2.p, ds.p, samples != nullptr, nullptr, n_draws, seed,
                        max_distance, confidence, max_trials, dm.p, dmi.p, dinl.p, dni.p, dacc.p, dused.p));
  APS_CUDA(cudaMemcpyAsync(models, dm.p, (size_t)n_pairs * 72, cudaMemcpyDeviceToHost, s));
  APS_CUDA(cudaMemcpyAsync(models_inv, dmi.p, (size_t)n_pairs * 72, cudaMemcpyDeviceToHost, s));
  if (total > 0) APS_CUDA(cudaMemcpyAsync(inliers, dinl.p, (size_t)total, cudaMemcpyDeviceToHost, s));
  APS_CUDA(cudaMemcpyAsync(n_inliers, dni.p, (size_t)n_pairs * 4, cudaMemcpyDeviceToHost, s));
  APS_CUDA(cudaMemcpyAsync(accepted, dacc.p, (size_t)n_pairs, cudaMemcpyDeviceToHost, s));
  APS_CUDA(cudaMemcpyAsync(draws_used, dused.p, (size_t)n_pairs * 4, cudaMemcpyDeviceToHost, s));
  APS_CUDA(cudaStreamSynchronize(s));
  return APS_OK;
}

extern "C" int aps_image_matching(aps_ctx* c, int n_images, const int64_t* pair_ptr, const uint32_t* rows,
                                  const double* keypoints, const int64_t* img_off, const int64_t* pairs_lin,
                                  int64_t n_pairs, double max_distance, double confidence, int max_trials,
                                  const uint32_t* samples, int64_t n_draws, uint64_t seed, int64_t* pt_ptr_out,
                                  double* models, double* models_inv, uint8_t* inliers, int32_t* n_inliers,
                                  uint8_t* accepted, int32_t* draws_used) {
  if (!c) APS_FAIL(APS_ERR_NOGPU, "apsmatch:nogpu", "context is NULL (no GPU context; there is no CPU path)");
  if (n_images < 0 || n_pairs < 0 || (n_pairs > 0 && (!pair_ptr || !pairs_lin || !img_off || !pt_ptr_out)))
    APS_FAIL(APS_ERR_ARGS, "", "bad arguments");
  if (n_pairs == 0) return APS_OK;
  std::vector<int64_t> ptr((size_t)n_pairs + 1, 0);
  std::vector<int32_t> ii((size_t)n_pairs), jj((size_t)n_pairs);
  for (int64_t p = 0; p < n_pairs; ++p) {
    const int64_t lin = pairs_lin[p];
    if (lin < 0 || lin >= (int64_t)n_images * n_images) APS_FAIL(APS_ERR_ARGS, "", "pair index out of range");
    ii[p] = (int32_t)(lin % n_images);
    jj[p] = (int32_t)(lin / n_images);
    ptr[p + 1] = ptr[p] + (pair_ptr[lin + 1] - pair_ptr[lin]);
  }
  for (int64_t p = 0; p <= n_pairs; ++p) pt_ptr_out[p] = ptr[p];
  APS_TRY(ransac_args(c, n_pairs, ptr.data(), n_draws, max_trials, confidence));
  APS_CUDA(cudaSetDevice(c->device));
  const int64_t total = ptr[n_pairs], F = img_off[n_images];
  if ((total > 0 && (!rows || !keypoints || !inliers)) || !models || !models_inv || !n_inliers || !accepted || !draws_used)
    APS_FAIL(APS_ERR_ARGS, "", "NULL argument");
  std::vector<uint32_t> crow((size_t)(2 * total));
  for (int64_t p = 0; p < n_pairs; ++p) {  // refineMatch:214-221: indices must lie inside the keypoint arrays
    const int64_t lin = pairs_lin[p], a = pair_ptr[lin], cntp = ptr[p + 1] - ptr[p];
    const int64_t ni = img_off[ii[p] + 1] - img_off[ii[p]], nj = img_off[jj[p] + 1] - img_off[jj[p]];
    for (int64_t r = 0; r < cntp; ++r) {
      const uint32_t ra = rows[2 * (a + r)], rb = rows[2 * (a + r) + 1];
      if (ra < 1 || rb < 1 || (int64_t)ra > ni || (int64_t)rb > nj)
        APS_FAIL(APS_ERR_ARGS, "refineMatch:MatchIndexOutOfBounds", "Match indices exceed keypoint array sizes.");
      crow[2 * (ptr[p] + r)] = ra;
      crow[2 * (ptr[p] + r) + 1] = rb;
    }
  }
  cudaStream_t s = c->stream;
  DevBuf<int64_t> dptr, doff;
  DevBuf<int32_t> dii, djj, dni, dused;
  DevBuf<uint32_t> drows, ds;
  DevBuf<double2> dkp, dp1, dp2;
  DevBuf<double> dm, dmi;
  DevBuf<uint8_t> dinl, dacc;
  const size_t tot = (size_t)(total > 0 ? total : 1);
  APS_TRY(dptr.alloc((size_t)n_pairs + 1, s));
  APS_TRY(doff.alloc((size_t)n_images + 1, s));
  APS_TRY(dii.alloc((size_t)n_pairs, s));
  APS_TRY(djj.alloc((size_t)n_pairs, s));
  APS_TRY(drows.alloc(2 * tot, s));
  APS_TRY(dkp.alloc((size_t)(F > 0 ? F : 1), s));
  APS_TRY(dp1.alloc(tot, s));
  APS_TRY(dp2.alloc(tot, s));
  APS_TRY(ds.alloc((size_t)(n_pairs * n_draws * 4), s));
  APS_TRY(dm.alloc((size_t)n_pairs * 9, s));
  APS_TRY(dmi.alloc((size_t)n_pairs * 9, s));
  APS_TRY(dinl.alloc(tot, s));
  APS_TRY(dacc.alloc((size_t)n_pairs, s));
  APS_TRY(dni.alloc((size_t)n_pairs, s));
  APS_TRY(dused.alloc((size_t)n_pairs, s));
  APS_CUDA(cudaMemcpyAsync(dptr.p, ptr.data(), (size_t)(n_pairs + 1) * 8, cudaMemcpyHostToDevice, s));
  APS_CUDA(cudaMemcpyAsync(doff.p, img_off, (size_t)(n_images + 1) * 8, cudaMemcpyHostToDevice, s));
  APS_CUDA(cudaMemcpyAsync(dii.p, ii.data(), (size_t)n_pairs * 4, cudaMemcpyHostToDevice, s));
  APS_CUDA(cudaMemcpyAsync(djj.p, jj.data(), (size_t)n_pairs * 4, cudaMemcpyHostToDevice, s));
  if (total > 0) {
    APS_CUDA(cudaMemcpyAsync(drows.p, crow.data(), (size_t)total * 8, cudaMemcpyHostToDevice, s));
    APS_CUDA(cudaMemcpyAsync(dkp.p, keypoints, (size_t)F * 16, cudaMemcpyHostToDevice, s));
    k_gather_matched_points<<<dim3(8, (unsigned)n_pairs), 256, 0, s>>>(dptr.p, drows.p, dii.p, djj.p, doff.p, dkp.p,
                                                                       dp1.p, dp2.p);
    APS_LAUNCHED();
  }
  if (samples)
    APS_CUDA(cudaMemcpyAsync(ds.p, samples, (size_t)(n_pairs * n_draws * 4) * 4, cudaMemcpyHostToDevice, s));
  APS_TRY(ransac_device(c, n_pairs, total, dptr.p, dp1.p, dp2.p, ds.p, samples != nullptr, nullptr, n_draws, seed,
                        max_distance, confidence, max_trials, dm.p, dmi.p, dinl.p, dni.p, dacc.p, dused.p));
  APS_CUDA(cudaMemcpyAsync(models, dm.p, (size_t)n_pairs * 72, cudaMemcpyDeviceToHost, s));
  APS_CUDA(cudaMemcpyAsync(models_inv, dmi.p, (size_t)n_pairs * 72, cudaMemcpyDeviceToHost, s));
  if (total > 0) APS_CUDA(cudaMemcpyAsync(inliers, dinl.p, (size_t)total, cudaMemcpyDeviceToHost, s));
  APS_CUDA(cudaMemcpyAsync(n_inliers, dni.p, (size_t)n_pairs * 4, cudaMemcpyDeviceToHost, s));
  APS_CUDA(cudaMemcpyAsync(accepted, dacc.p, (size_t)n_pairs, cudaMemcpyDeviceToHost, s));
  APS_CUDA(cudaMemcpyAsync(draws_used, dused.p, (size_t)n_pairs * 4, cudaMemcpyDeviceToHost, s));
  APS_CUDA(cudaStreamSynchronize(s));  // crow / ptr / ii / jj stay alive until here
  return APS_OK;
}

// imageMatching.m:121-156 for every candidate pair of nsets image sets.  Set b's pairs are
// set_pair_ptr[b] .. set_pair_ptr[b + 1] of pairs_lin (cells of its own n_b x n_b block); its images are the pooled
// images g_b .. g_b + n_b of img_off / keypoints.  Pair p of set b draws its samples under key p - set_pair_ptr[b], the
// key its single-set call gives it, so every set gets the single-set call's bits.  The gather and the RANSAC chain
// run in chunks of pairs: gridDim.y holds at most 65535 pairs, and the per-draw tables (kSetsDrawBytes per draw and
// pair) stay within kSetsChunkBytes.  pt_ptr offsets are absolute, so a chunk only offsets the per-pair pointers.
static constexpr int64_t kSetsDrawBytes = 16 + 72 + 4 + 8;  // sample table, Htab, cnt, err
static constexpr int64_t kSetsChunkBytes = (int64_t)1 << 30;

extern "C" int aps_image_matching_sets(aps_ctx* c, int nsets, const int* set_images, const int64_t* const* pair_ptr,
                                       const uint32_t* const* rows, const double* keypoints, const int64_t* img_off,
                                       const int64_t* set_pair_ptr, const int64_t* pairs_lin, double max_distance,
                                       double confidence, int max_trials, const uint32_t* samples, int64_t n_draws,
                                       uint64_t seed, int64_t* pt_ptr_out, double* models, double* models_inv,
                                       uint8_t* inliers, int32_t* n_inliers, uint8_t* accepted, int32_t* draws_used) {
  if (nsets < 0 || (nsets > 0 && (!set_images || !set_pair_ptr))) APS_FAIL(APS_ERR_ARGS, "", "bad set list");
  std::vector<int64_t> img0((size_t)nsets + 1, 0);
  for (int b = 0; b < nsets; ++b) {
    if (set_images[b] < 0) APS_FAIL(APS_ERR_ARGS, "", "set %d: negative image count", b + 1);
    img0[b + 1] = img0[b] + set_images[b];
  }
  if (img0[nsets] > INT32_MAX) APS_FAIL(APS_ERR_ARGS, "", "more than 2^31 - 1 images");
  if (nsets > 0 && set_pair_ptr[0] != 0) APS_FAIL(APS_ERR_ARGS, "", "set_pair_ptr[0] must be 0");
  for (int b = 0; b < nsets; ++b)
    if (set_pair_ptr[b + 1] < set_pair_ptr[b]) APS_FAIL(APS_ERR_ARGS, "", "set_pair_ptr must be non-decreasing");
  APS_TRY(ransac_params(n_draws, max_trials, confidence));
  const int64_t n_pairs = nsets > 0 ? set_pair_ptr[nsets] : 0, G = img0[nsets];
  if (n_pairs > 0 && (!pair_ptr || !rows || !pairs_lin || !img_off || !pt_ptr_out || !models || !models_inv ||
                      !n_inliers || !accepted || !draws_used))
    APS_FAIL(APS_ERR_ARGS, "", "NULL argument");
  std::vector<int64_t> ptr((size_t)n_pairs + 1, 0), keys((size_t)n_pairs);
  std::vector<int32_t> ii((size_t)n_pairs), jj((size_t)n_pairs);
  for (int b = 0; b < nsets; ++b) {
    const int64_t n = set_images[b];
    for (int64_t p = set_pair_ptr[b]; p < set_pair_ptr[b + 1]; ++p) {
      const int64_t lin = pairs_lin[p];
      if (!pair_ptr[b] || lin < 0 || lin >= n * n) APS_FAIL(APS_ERR_ARGS, "", "set %d: pair index out of range", b + 1);
      const int64_t cnt = pair_ptr[b][lin + 1] - pair_ptr[b][lin];
      if (cnt < 0) APS_FAIL(APS_ERR_ARGS, "", "set %d: pair_ptr must be non-decreasing", b + 1);
      ii[p] = (int32_t)(img0[b] + lin % n);
      jj[p] = (int32_t)(img0[b] + lin / n);
      keys[p] = p - set_pair_ptr[b];
      ptr[p + 1] = ptr[p] + cnt;
    }
  }
  const int64_t total = ptr[n_pairs], F = n_pairs > 0 ? img_off[G] : 0;
  if (total > 0 && (!keypoints || !inliers)) APS_FAIL(APS_ERR_ARGS, "", "NULL argument");
  std::vector<uint32_t> crow((size_t)(2 * total));
  for (int b = 0; b < nsets; ++b)
    for (int64_t p = set_pair_ptr[b]; p < set_pair_ptr[b + 1]; ++p) {  // refineMatch:214-221
      const int64_t a = pair_ptr[b][pairs_lin[p]], cntp = ptr[p + 1] - ptr[p];
      const int64_t ni = img_off[ii[p] + 1] - img_off[ii[p]], nj = img_off[jj[p] + 1] - img_off[jj[p]];
      if (cntp > 0 && !rows[b]) APS_FAIL(APS_ERR_ARGS, "", "set %d: rows is NULL", b + 1);
      for (int64_t r = 0; r < cntp; ++r) {
        const uint32_t ra = rows[b][2 * (a + r)], rb = rows[b][2 * (a + r) + 1];
        if (ra < 1 || rb < 1 || (int64_t)ra > ni || (int64_t)rb > nj)
          APS_FAIL(APS_ERR_ARGS, "refineMatch:MatchIndexOutOfBounds",
                   "Match indices exceed keypoint array sizes (set %d).", b + 1);
        crow[2 * (ptr[p] + r)] = ra;
        crow[2 * (ptr[p] + r) + 1] = rb;
      }
    }
  if (!c) APS_FAIL(APS_ERR_NOGPU, "apsmatch:nogpu", "context is NULL (no GPU context; there is no CPU path)");
  APS_CUDA(cudaSetDevice(c->device));
  if (pt_ptr_out)
    for (int64_t p = 0; p <= n_pairs; ++p) pt_ptr_out[p] = ptr[p];
  if (n_pairs == 0) return APS_OK;
  const int64_t by_bytes = kSetsChunkBytes / (n_draws * kSetsDrawBytes);
  const int64_t chunk = aps_min64(65535, by_bytes > 0 ? by_bytes : 1);
  cudaStream_t s = c->stream;
  DevBuf<int64_t> dptr, doff, dkeys;
  DevBuf<int32_t> dii, djj, dni, dused;
  DevBuf<uint32_t> drows, ds;
  DevBuf<double2> dkp, dp1, dp2;
  DevBuf<double> dm, dmi;
  DevBuf<uint8_t> dinl, dacc;
  const size_t tot = (size_t)(total > 0 ? total : 1);
  APS_TRY(dptr.alloc((size_t)n_pairs + 1, s));
  APS_TRY(doff.alloc((size_t)G + 1, s));
  APS_TRY(dkeys.alloc((size_t)n_pairs, s));
  APS_TRY(dii.alloc((size_t)n_pairs, s));
  APS_TRY(djj.alloc((size_t)n_pairs, s));
  APS_TRY(drows.alloc(2 * tot, s));
  APS_TRY(dkp.alloc((size_t)(F > 0 ? F : 1), s));
  APS_TRY(dp1.alloc(tot, s));
  APS_TRY(dp2.alloc(tot, s));
  APS_TRY(ds.alloc((size_t)(aps_min64(chunk, n_pairs) * n_draws * 4), s));
  APS_TRY(dm.alloc((size_t)n_pairs * 9, s));
  APS_TRY(dmi.alloc((size_t)n_pairs * 9, s));
  APS_TRY(dinl.alloc(tot, s));
  APS_TRY(dacc.alloc((size_t)n_pairs, s));
  APS_TRY(dni.alloc((size_t)n_pairs, s));
  APS_TRY(dused.alloc((size_t)n_pairs, s));
  APS_CUDA(cudaMemcpyAsync(dptr.p, ptr.data(), (size_t)(n_pairs + 1) * 8, cudaMemcpyHostToDevice, s));
  APS_CUDA(cudaMemcpyAsync(doff.p, img_off, (size_t)(G + 1) * 8, cudaMemcpyHostToDevice, s));
  APS_CUDA(cudaMemcpyAsync(dkeys.p, keys.data(), (size_t)n_pairs * 8, cudaMemcpyHostToDevice, s));
  APS_CUDA(cudaMemcpyAsync(dii.p, ii.data(), (size_t)n_pairs * 4, cudaMemcpyHostToDevice, s));
  APS_CUDA(cudaMemcpyAsync(djj.p, jj.data(), (size_t)n_pairs * 4, cudaMemcpyHostToDevice, s));
  if (total > 0) {
    APS_CUDA(cudaMemcpyAsync(drows.p, crow.data(), (size_t)total * 8, cudaMemcpyHostToDevice, s));
    APS_CUDA(cudaMemcpyAsync(dkp.p, keypoints, (size_t)F * 16, cudaMemcpyHostToDevice, s));
  }
  for (int64_t p0 = 0; p0 < n_pairs; p0 += chunk) {
    const int64_t np = aps_min64(chunk, n_pairs - p0);
    if (ptr[p0 + np] > ptr[p0]) {
      k_gather_matched_points<<<dim3(8, (unsigned)np), 256, 0, s>>>(dptr.p + p0, drows.p, dii.p + p0, djj.p + p0, doff.p,
                                                                    dkp.p, dp1.p, dp2.p);
      APS_LAUNCHED();
    }
    if (samples)
      APS_CUDA(cudaMemcpyAsync(ds.p, samples + p0 * n_draws * 4, (size_t)(np * n_draws * 4) * 4, cudaMemcpyHostToDevice,
                               s));
    APS_TRY(ransac_device(c, np, total, dptr.p + p0, dp1.p, dp2.p, ds.p, samples != nullptr, dkeys.p + p0, n_draws, seed,
                          max_distance, confidence, max_trials, dm.p + 9 * p0, dmi.p + 9 * p0, dinl.p, dni.p + p0,
                          dacc.p + p0, dused.p + p0));
  }
  APS_CUDA(cudaMemcpyAsync(models, dm.p, (size_t)n_pairs * 72, cudaMemcpyDeviceToHost, s));
  APS_CUDA(cudaMemcpyAsync(models_inv, dmi.p, (size_t)n_pairs * 72, cudaMemcpyDeviceToHost, s));
  if (total > 0) APS_CUDA(cudaMemcpyAsync(inliers, dinl.p, (size_t)total, cudaMemcpyDeviceToHost, s));
  APS_CUDA(cudaMemcpyAsync(n_inliers, dni.p, (size_t)n_pairs * 4, cudaMemcpyDeviceToHost, s));
  APS_CUDA(cudaMemcpyAsync(accepted, dacc.p, (size_t)n_pairs, cudaMemcpyDeviceToHost, s));
  APS_CUDA(cudaMemcpyAsync(draws_used, dused.p, (size_t)n_pairs * 4, cudaMemcpyDeviceToHost, s));
  APS_CUDA(cudaStreamSynchronize(s));  // crow / ptr / keys / ii / jj stay alive until here
  return APS_OK;
}
