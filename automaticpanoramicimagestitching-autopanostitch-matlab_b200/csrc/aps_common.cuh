// aps_common.cuh -- shared declarations of libapsmatch (B200 / sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <vector>

#include "../../include/apsmatch.h"

#define APS_EPS32 1.1920928955078125e-07f  // eps('single')

void aps_set_error(int code, const char* id, const char* fmt, ...);
void aps_count_launch(int n = 1);  // every kernel launch of the library is counted (bench.py's gpu_launches)

#define APS_CUDA(call)                                                                                        \
  do {                                                                                                        \
    cudaError_t e__ = (call);                                                                                 \
    if (e__ != cudaSuccess) {                                                                                 \
      aps_set_error(APS_ERR_CUDA, "", "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__,     \
                    __LINE__);                                                                                \
      return APS_ERR_CUDA;                                                                                    \
    }                                                                                                         \
  } while (0)

// after every <<<>>> launch: count it and check the launch status
#define APS_LAUNCHED()       \
  do {                       \
    aps_count_launch();      \
    APS_CUDA(cudaGetLastError()); \
  } while (0)

#define APS_TRY(call)          \
  do {                         \
    int rc__ = (call);         \
    if (rc__ != APS_OK) return rc__; \
  } while (0)

struct aps_ctx {
  int device = 0;
  int sm_count = 148;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  int float_engine = 0;  // 0 auto, 1 exact only, 2 tensor required
  int pairwise_screen = 1;     // 1: fp16 tensor screen before the exact pairwise pipeline (aps_pair_screen.cu), 0: off
  int64_t pair_stats[4] = {0, 0, 0, 0};  // last pairwise match: pairs screened, pairs surviving, entries screened, -
  int pairwise_epilogue = -1;  // -1 auto, 0 streaming top-4, 1 branch-free segment selection (aps_ctx_set_pairwise_epilogue)
  int64_t stats[4] = {0, 0, 0, 0};
  bool timing = false;
  std::vector<cudaEvent_t> tc_events;  // pairs (start, stop) of tcgen05 kernel launches
  int32_t* d_scratch_flags = nullptr;  // small persistent device scratch (64 ints)
  int32_t* h_flags = nullptr;          // pinned mirror
  void* h_stage = nullptr;             // grow-only pinned staging area for result downloads (aps_ctx_stage)
  size_t h_stage_bytes = 0;
};
// pinned host staging of at least `bytes` (contents undefined); nullptr on allocation failure
inline void* aps_ctx_stage(aps_ctx* c, size_t bytes) {
  if (bytes <= c->h_stage_bytes) return c->h_stage;
  if (c->h_stage) cudaFreeHost(c->h_stage);
  c->h_stage = nullptr;
  c->h_stage_bytes = 0;
  const size_t want = bytes + bytes / 4 + 4096;
  if (cudaMallocHost(&c->h_stage, want) != cudaSuccess) { c->h_stage = nullptr; (void)cudaGetLastError(); return nullptr; }
  c->h_stage_bytes = want;
  return c->h_stage;
}

// Stream-ordered device buffer (cudaMallocAsync pool: repeated calls re-use the same memory).
template <class T>
struct DevBuf {
  T* p = nullptr;
  size_t n = 0;
  cudaStream_t s = nullptr;
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() { release(); }
  int alloc(size_t count, cudaStream_t stream) {
    release();
    s = stream;
    n = count;
    if (count == 0) return APS_OK;
    cudaError_t e = cudaMallocAsync((void**)&p, count * sizeof(T), stream);
    if (e != cudaSuccess) {
      p = nullptr;
      aps_set_error(APS_ERR_ALLOC, "", "cudaMallocAsync(%zu bytes) failed: %s", count * sizeof(T),
                    cudaGetErrorString(e));
      return APS_ERR_ALLOC;
    }
    return APS_OK;
  }
  void release() {
    if (p) cudaFreeAsync(p, s);
    p = nullptr;
    n = 0;
  }
};

static inline int64_t aps_ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }
static inline int64_t aps_min64(int64_t a, int64_t b) { return a < b ? a : b; }

// ---- kernel launchers (one translation unit each) ------------------------------------------
// K1  aps_prep.cu
enum { APS_NORM_NONE = 0, APS_NORM_GLOBAL = 1, APS_NORM_PAIRWISE = 2 };
// transposes one image's column-major [N x D] block into rows [row0,row0+N) of the row-major pool
int aps_k_transpose_in(cudaStream_t s, const void* src_cm, int64_t N, int D, int elem_size, void* dst_rm);
int aps_k_transpose_out_u32f32(cudaStream_t s, const uint32_t* idx_rm, const float* dist_rm, int64_t N, int k,
                               uint32_t* idx_cm, float* dist_cm);
// pass 1: xn = normalised rows (norm_mode), sq[r] = sum(xn^2) (sequential f32), invn[r] = 1/norm (1 when
// norm_mode NONE), flags[0] &= all raw values exactly representable in bf16, flags[1] = max bits |sq-1|,
// flags[2] = max bits sq, flags[3] = max bits |raw| (for the max|.|>2 test of matchFeaturesScratch.m:105)
// fp16 = 1: flags[0] speaks about exact representability in fp16 (the operand type the caller will build)
int aps_k_prepare_norm(cudaStream_t s, const float* raw, int64_t F, int D, int norm_mode, float* xn, float* sq,
                       float* invn, int32_t* flags, int fp16 = 0);
// the same for every image of a pooled matrix in one launch: image i = rows [img_off[i], img_off[i+1]), flags + 8*i
int aps_k_prepare_norm_images(cudaStream_t s, const float* raw, const int64_t* d_img_off, int n, int64_t maxcount, int D,
                              int norm_mode, float* xn, float* sq, float* invn, int32_t* flags, int fp16 = 0);
// pass 2: bf16 operands [F x Dp] (Dp multiple of 64, zero padded) + per-column (scale,bias)
//   exact_flag (device int): 1 -> operand = bf16(raw), scale = invn ; 0 -> operand = bf16(xn), scale = 1
//   bias_mode: 0 -> bias 0 ; 1 -> bias = -sq/2 (SSD on un-normalised rows)
int aps_k_prepare_operands(cudaStream_t s, const float* raw, const float* xn, const float* sq, const float* invn,
                           int64_t F, int D, int Dp, const int32_t* exact_flag, int bias_mode, __nv_bfloat16* xb,
                           float* colscale, float* colbias, int fp16 = 0);  // fp16 = 1: the rows are written as fp16

// train-side view of the tensor kernel (aps_prep.cu)
int aps_k_sort_train_by_scale(cudaStream_t s, const __nv_bfloat16* xb, const float* colscale, const float* colbias,
                              int64_t N, int Dp, int32_t* scratch, int32_t* perm, __nv_bfloat16* xb_t,
                              float* colscale_t, float* colbias_t);
int aps_sort_scratch_ints();
int aps_k_tile_bounds(cudaStream_t s, const float* colscale, const float* colbias, int64_t N, int tile_rows,
                      float4* out);

// K2f aps_knn_exact.cu : exact CUDA-core kNN.  rows==nullptr -> queries [q0,q0+nq) ; else rows[i].
//   metric 0: FLANN-order squared L2 ; metric 1: SSD order (a2 + b2) - 2*G with sq arrays.
//   train columns [t0,t1) ; output idx 1-based RELATIVE TO t0 (idx = j - t0 + 1), row-major [.. x k],
//   written at out row = (rows ? rows[i] : q0 + i) - out_row0.
int aps_k_knn_exact(cudaStream_t s, const float* Q, const float* sqQ, const int32_t* rows, const int32_t* nrows_dev,
                    int64_t q0, int64_t nq, const float* T, const float* sqT, int64_t t0, int64_t t1, int D,
                    int k, int metric, int64_t out_row0, uint32_t* idx, float* dist);
// set-restricted search of the pooled rows X [F x D] (metric 0): group table {row0, rows <= 8, t0, t1} per CTA task,
// neighbour indices 1-based over all F rows; ngroups_dev (optional): device-side group count (<= ngroups)
int aps_k_knn_exact_groups(cudaStream_t s, const float* X, const int4* d_groups, int64_t ngroups,
                           const int32_t* ngroups_dev, int D, int k, uint32_t* idx, float* dist);
constexpr int APS_EXACT_GROUP_ROWS = 8;

// K4 aps_hamming.cu : exact Hamming kNN, thread per query, k <= APS_MAX_K.  idx relative to t0, 1-based.
int aps_k_knn_hamming(cudaStream_t s, const uint8_t* Q, int64_t q0, int64_t nq, const uint8_t* T, int64_t t0,
                      int64_t t1, int nb, int k, int64_t out_row0, uint32_t* idx, float* dist);
// set-restricted Hamming search: one CTA per group {row0, rows <= aps_k_knn_hamming_group_rows(), t0, t1}
int aps_k_knn_hamming_groups(cudaStream_t s, const uint8_t* X, const int4* d_groups, int64_t ngroups, int nb16, int k,
                             uint32_t* idx, float* dist);
int aps_k_knn_hamming_group_rows();

// K2 aps_knn_tc.cu : tcgen05 candidate search.  See the file header.
struct aps_tc_unit {  // explicit work unit of the batched launch
  int32_t qrow0;    // first query row (global) of a block of up to 256 rows
  int32_t qend;     // one past the last query row that belongs to the unit
  int32_t t0, t1;   // train rows searched
  int64_t out_row;  // row of qrow0 in the candidate buffers
};
struct aps_tc_problem {
  const __nv_bfloat16* Qb;  // [Fq_total x Dp] query operands
  const __nv_bfloat16* Tb;  // [Ft_total x Dp] train operands
  const float* colscale;    // [Ft_total + 256] per train row
  const float* colbias;     // [Ft_total + 256] per train row (used iff bias)
  const float4* tile_bounds;  // per 128-row tile of Tb: (1/scale_max, 1/scale_min, bias_max, -)
  int bias;                 // 0: score = dot*scale ; 1: score = dot*scale + bias
  int64_t Fq_total, Ft_total;
  int Dp;
  int64_t q0, q1;  // query rows to search
  int64_t t0, t1;  // train rows searched
  int nslot;       // candidate lists per row: aps_k_knn_tc_slots(...) for this problem
  int kcand;       // candidates kept per (row, segment): 8 (k <= 5) or 16 (6 <= k <= 12)
  uint32_t* cand_idx;   // [ (q1-q0) x nslot x kcand ] global train row (0-based) or 0xFFFFFFFF
  float* cand_score;    // same shape: score (dot*scale+bias), -inf for empty slots
  float* dump;          // optional [ (q1-q0) x (t1-t0) ] raw scores (tests only), else nullptr
  const int32_t* nrows_dev = nullptr;  // second pass: Qb holds *nrows_dev gathered rows (q0 = 0, q1 = upper bound)
  int operand_fp16 = 0;                // != 0: Qb / Tb hold fp16 rows (|x| within the fp16 range): kind::f16 with F16 inputs,
                                       // F32 accumulate.  1 = operands never treated as exact, 2 = flags[0] says whether they are
  const int32_t* exact_flag = nullptr; // device flag "operands are exact in bf16" (K1): when given, the first pass keeps 6
                                       // candidates per list instead of 8 for exact operands (lists stay 8 wide, two
                                       // entries empty): eps is ~1e-4 then, and 6 still prove a top-5.  Not read
                                       // with kcand 16
};
int aps_k_knn_tc_supported(int Dp);
int aps_k_knn_tc_tile_rows();  // rows per train tile (for aps_k_tile_bounds)
int aps_k_knn_tc_tile_mode_stride();   // unit-table launch with kcand == 3: candidate entries per row (2 lists x 3)
int aps_k_knn_tc_tile_mode_segment();  // ... and the columns per segment (two best kept per segment)
int aps_k_knn_tc_units(cudaStream_t s, int sm_count, const aps_tc_problem& p, const aps_tc_unit* d_units,
                       int64_t n_units);
int aps_k_knn_tc_slots(int sm_count, int64_t nq, int64_t t0, int64_t t1, int all_segmented = 0);  // lists per row
// the schedule aps_k_knn_tc launches for p: out[0..6] = nslot, pre-filtered long sweep (0/1), units_full, tail_units,
// tail_seg, tail_balanced, tiles_per_seg
int aps_k_knn_tc_describe(int sm_count, const aps_tc_problem& p, int* out);
int64_t aps_k_knn_tc_full_rows(int sm_count, int64_t nq, int64_t t0, int64_t t1);  // leading query rows that only fill list 0
int aps_k_gather_rows(cudaStream_t s, const __nv_bfloat16* src, int Dp, const int32_t* rows, const int32_t* nrows_dev,
                      int64_t max_rows, __nv_bfloat16* dst);
// ev0/ev1 (optional): recorded immediately before / after the candidate kernel itself
int aps_k_knn_tc(cudaStream_t s, int sm_count, const aps_tc_problem& p, cudaEvent_t ev0 = nullptr,
                 cudaEvent_t ev1 = nullptr);

// batched pairwise bookkeeping: entry e of pair p (eoff[p] <= e < eoff[p+1]) is query row qoff[p] + e - eoff[p]
// searched in train rows [toff[p], toff[p] + tcnt[p])
struct aps_pair_tables {
  const int64_t* eoff;   // [npairs + 1] entry offsets
  const int32_t* qoff;   // [npairs] first global row of the query image
  const int32_t* toff;   // [npairs] first global row of the train image
  const int32_t* tcnt;   // [npairs] rows of the train image
  const int64_t* boff;   // [npairs + 1] offsets into per-train-row scratch (sum of tcnt)
  int npairs;
  // K3 shortcut for the batched pairwise path: a query whose APPROXIMATE best / second-best distances already
  // prove that matchFeaturesScratch.m:174-178 rejects it (d1 > r2*d2 or d1 > MatchThreshold, with the eps
  // margin on both sides) is written as "no neighbour" without recomputing exact distances.
  int prune;
  double prune_r2, prune_mt;
  // > 0: the candidate lists come from the branch-free segment epilogue (k_knn_tc<.., 3, 2>): each list holds the
  // three best of "two best per segment of tile_mode columns", sorted by approximate score.  A column outside a list
  // is then bounded by the list's third entry -- or by its second when the two best share a segment -- and eps
  // grows by the 7 key bits.
  int tile_mode;
  // != 0: the tensor pass ran on fp16 operands (10-bit mantissa): the operand-rounding term of eps is 2.0e-3 instead of
  // 1.57e-2.  1 = never exact (pairwise: normalised rows are rounded), 2 = flags[0] tells (global path, set by K1)
  int operand_fp16;
  // 'subsetpdist2' with images above the subset size: the train rows of such an image are a random subset stored as a
  // "virtual image" at rows >= vfirst of the train view; vmap[row - vfirst] = 0-based local index in the original image
  const int32_t* vmap;
  int64_t vfirst;
};

// aps_pair_screen.cu : pairwise stage 1 -- fp16 tensor-core screen of every (query row, train image); see the file header
struct aps_pair_screen_tables {   // per image pair p of the launch (device arrays)
  const int32_t* qoff;   // first global row of the query image
  const int32_t* qcnt;   // rows of the query image
  const int32_t* toff;   // first global row of the train image
  const int32_t* tcnt;   // rows of the train image
  const int32_t* timg;   // train image index (per-image norm bounds)
  const int64_t* eoff;   // [npairs + 1] entry offsets (sum of qcnt)
  const int64_t* uoff;   // [npairs + 1] unit offsets (sum of ceil(qcnt / 256))
  int npairs;
};
// bound of |fp16 tensor dot - exact dot| in units of |a||b|: operand rounding 2 * 2^-11, one rounding of the running
// sum to fp16 per K = 16 instruction (2^-10 each, Dp / 16 of them), margin.  Checked against measurements by
// tests/test_gpu_pair_screen.py.
__host__ __device__ inline float aps_pair_screen_dot_eps(int Dp) { return (float)(Dp / 16) * 9.765625e-4f + 1.5e-3f; }
int aps_k_fill_f32(cudaStream_t s, float* dst, int64_t n, float v);
int aps_k_prepare_operands_f16(cudaStream_t s, const float* src, int64_t F, int D, int Dp, void* xh);
// per train image i: (min, max) of sq over rows [start[i], start[i] + count[i])
int aps_k_image_sq_bounds(cudaStream_t s, const float* sq, const int64_t* d_start, const int64_t* d_count, int n, float2* out);
// xh_q / xh_t: fp16 operand rows of the query side [Fq x Dp] and of the train view [Ft x Dp] (the same matrix unless
// the train view carries subset images)
int aps_k_pair_screen(cudaStream_t s, int sm_count, const void* xh_q, int64_t Fq, const void* xh_t, int64_t Ft, int Dp,
                      const aps_pair_screen_tables& t, aps_tc_unit* d_units, int64_t n_units, uint32_t* out,
                      uint32_t* dump = nullptr, int dump_tiles = 0);
// virtual (subset) images: vsrc[v] = global source row of virtual row v, chosen by a keyed bijection of [0, N_j) whose
// key is (seed, d_key_img[b]) for big image b = d_big_img[b]
int aps_k_subset_rows(cudaStream_t s, const int64_t* d_img_off, const int32_t* d_big_img, const int32_t* d_key_img,
                      int nbig, int64_t subset, uint64_t seed, int32_t* vsrc, int32_t* vmap);
int aps_k_gather_f32_rows(cudaStream_t s, const float* src, const int32_t* rows, int64_t nrows, int D, float* dst);
int aps_k_gather_u16_rows(cudaStream_t s, const uint16_t* src, const int32_t* rows, int64_t nrows, int Dp, uint16_t* dst);
int aps_k_pair_screen_decide(cudaStream_t s, const uint32_t* scr, const float* sq, const aps_pair_screen_tables& t,
                             const float2* img_bounds, const int32_t* flags, int Dp, double r2, double mt,
                             int32_t* survivors);

// aps_pca.cu : 'pca2nn' front end (mean, covariance, Jacobi eigenvectors per image; table-driven projections)
struct aps_proj_seg {   // rows [src, src + cnt) of X projected with the basis of image `basis` into rows [dst, dst + cnt)
  int64_t src, dst;
  int32_t cnt, basis;
};
int aps_pca_components();
int aps_k_pca_basis(cudaStream_t s, const float* X, const int64_t* d_img_off, int n, int D, int P, float* mu, float* coeff,
                    double* scratch /* 2 * n * D * D */);
int aps_k_pca_project(cudaStream_t s, const float* X, int D, int P, const std::vector<aps_proj_seg>& segs, const float* mu,
                      const float* coeff, float* out);

// K3 aps_rerank.cu : exact FP32 re-rank of the candidates + completeness proof.
//   approx distance of a score: alpha[row] + beta[row]*score ; row proven iff
//   (worst retained approx distance over segments) - eps_bound > exact k-th distance.
//   Unproven rows are appended to fb_rows/fb_count for the exact kernel.
int aps_k_rerank(cudaStream_t s, const float* Q, const float* sqQ, const float* invnQ, const float* T,
                 const float* sqT, int D, int metric, int64_t q0, int64_t nq, int64_t t0, int nseg, int kcand,
                 const uint32_t* cand_idx, const float* cand_score, const int32_t* exact_flag, int bias_mode,
                 const int32_t* flags, int k, int64_t out_row0, uint32_t* idx, float* dist, int32_t* fb_rows,
                 int32_t* fb_count, const aps_pair_tables* pairs = nullptr, const int32_t* row_map = nullptr,
                 const int32_t* nrows_dev = nullptr, const int32_t* perm = nullptr, int cand_stride = 0,
                 int kcap_exact = 0);  // > 0: lists hold only this many entries when flags[0] (exact operands) is set

// K5 aps_filter.cu
int aps_k_global_filter(cudaStream_t s, const uint32_t* idx, const float* dist, int k, int64_t q0, int64_t q1,
                        const int32_t* img_of_row, const int64_t* img_off, float ratio_thr, int2* records);
int aps_k_records_mutual(cudaStream_t s, int2* records, const int32_t* img_of_row, const int64_t* img_off, int64_t F,
                         uint8_t* keep /* [F] scratch */);
// compaction of per-query records into the CSR cell order (featureMatchingGlobal.m:149-159)
int aps_k_fill_img_of_row(cudaStream_t s, const int64_t* img_off, int n, int64_t maxcount, int32_t* img_of_row);
int aps_k_global_compact(cudaStream_t s, const int2* records /* [F]: (target image + 1 | 0, partner) */,
                         const int32_t* img_of_row, const int64_t* img_off, int n, int64_t F, int64_t* dir_counts /*n*n*/,
                         int64_t* pair_counts /*n*n*/, int64_t* pair_ptr /*n*n+1*/, int64_t* rank /*F*/,
                         uint32_t* rows /*2F*/);
// the same over independent image sets: set s owns the cells [cell_off[s], cell_off[s] + n_s^2) (its own n_s x n_s
// block), so the tables hold sum(n_s^2) cells; one scan over all of them
int aps_k_global_compact_sets(cudaStream_t s, const int2* records, const int32_t* img_of_row, const int64_t* img_off,
                              int nimg, int64_t F, const int32_t* img_set, const int32_t* set_img0, const int32_t* set_n,
                              const int64_t* cell_off, int nsets, int max_n, int64_t cells, int64_t* dir_counts,
                              int64_t* pair_counts, int64_t* pair_ptr, int64_t* rank, uint32_t* rows);
int aps_k_hamming2_finalize(cudaStream_t s, int64_t N1, int64_t N2, int nb, const uint32_t* idx_k2,
                            const float* dist_k2, uint32_t* idx2, float* d1, float* d2);
int aps_k_split_k2(cudaStream_t s, int64_t N1, const uint32_t* idx_k2, const float* dist_k2, uint32_t* idx2,
                   float* d1, float* d2);
// pairwise: ratio/threshold filter + unique + sort for one (query image, train image) pair
int aps_k_pair_filter_unique(cudaStream_t s, const uint32_t* idx2, const float* d1, const float* d2, int64_t N1,
                             int64_t N2, int is_binary, int nbits, double match_threshold, double max_ratio,
                             int unique, unsigned long long* best_by_train /*N2*/, unsigned long long* keys /*2*N1*/,
                             int32_t* count_dev, uint32_t* matches /*2*N1*/, double* metric /*N1*/);

// K6 aps_select.cu
int aps_k_select_partners(cudaStream_t s, const int64_t* counts_cm, int n, int m, uint8_t* cand_cm);
// the same for nsets image sets: n_rows = sum n_b pooled images, set_img / cell_off [nsets + 1] = first pooled image and
// first cell of each set's n_b x n_b column-major block (cells = cell_off[nsets])
int aps_k_select_partners_sets(cudaStream_t s, const int64_t* counts, int n_rows, int64_t cells, const int64_t* set_img,
                               const int64_t* cell_off, int nsets, int m, uint8_t* cand);
// find() of every set's block: pairs_lin = cell indices inside the set's block, set-major; set_pair_ptr [nsets + 1]
int aps_k_select_compact(cudaStream_t s, const uint8_t* cand, int64_t cells, const int64_t* cell_off, int nsets,
                         int64_t* pairs_lin, int64_t* set_pair_ptr);

// aps_pairwise.cu : batched pairwise stages (see the file header)
// X / sq: query rows ; XT / sqT: train view (the same arrays unless the train view carries subset images)
int aps_k_pair_exact2(cudaStream_t s, const float* X, const float* sq, const float* XT, const float* sqT, int D, int metric,
                      const aps_pair_tables& pt, const int32_t* rows, const int32_t* nrows_dev, int64_t n_entries,
                      uint32_t* idx, float* dist);
int aps_k_pairs_hamming2(cudaStream_t s, const uint8_t* Xpad, int nb16, const std::vector<int64_t>& eoff,
                         const std::vector<int32_t>& qoff, const std::vector<int32_t>& toff,
                         const std::vector<int32_t>& tcnt, uint32_t* idx, float* dist);
int aps_k_pairs_k2_to_nn(cudaStream_t s, const aps_pair_tables& pt, int64_t E, int is_binary, int nb, const uint32_t* i2,
                         const float* dd, uint32_t* idx2, float* d1, float* d2);
int aps_k_pairs_filter_unique(cudaStream_t s, const aps_pair_tables& pt, int64_t E, int64_t Btotal,
                              const uint32_t* idx2, const float* d1, const float* d2, int is_binary, int nbits,
                              double match_threshold, double max_ratio, unsigned long long* best,
                              unsigned long long* keys, unsigned long long* winners, int32_t* count, uint32_t* matches,
                              double* metric);
