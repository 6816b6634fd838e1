// aps_abi.cu -- the extern "C" surface declared in include/apsmatch.h: argument checks with the
// reference's error identifiers, host<->device staging, and the kernel pipelines.
// No CPU compute path exists here: without a CUDA device every entry fails with APS_ERR_NOGPU.
#include <algorithm>
#include <atomic>
#include <cmath>
#include <limits>
#include <new>
#include <string>

#include "aps_abi_internal.cuh"

// ------------------------------------------------------------------------------------------------
// errors
static thread_local std::string g_err_msg;
static thread_local std::string g_err_id;

void aps_set_error(int code, const char* id, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err_msg = buf;
  g_err_id = id ? id : "";
  (void)code;
}

static std::atomic<int64_t> g_launches{0};
void aps_count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }
extern "C" int64_t aps_launch_count(void) { return g_launches.load(); }

extern "C" const char* aps_last_error(void) { return g_err_msg.c_str(); }
extern "C" const char* aps_error_id(void) { return g_err_id.c_str(); }
extern "C" int aps_abi_version(void) { return APS_ABI_VERSION; }


// ------------------------------------------------------------------------------------------------
// context
extern "C" int aps_ctx_create(int device, aps_ctx** out) {
  if (!out) APS_FAIL(APS_ERR_ARGS, "", "aps_ctx_create: out is NULL");
  *out = nullptr;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    APS_FAIL(APS_ERR_NOGPU, "apsmatch:nogpu",
             "no CUDA device available (%s); libapsmatch has no CPU fallback",
             e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
  if (device < 0 || device >= ndev) APS_FAIL(APS_ERR_ARGS, "", "device %d out of range (0..%d)", device, ndev - 1);
  APS_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  APS_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10)
    APS_FAIL(APS_ERR_NOGPU, "apsmatch:nogpu", "device %d is sm_%d%d; libapsmatch is built for sm_100a (B200) only",
             device, prop.major, prop.minor);
  aps_ctx* c = new (std::nothrow) aps_ctx();
  if (!c) APS_FAIL(APS_ERR_ALLOC, "", "out of host memory");
  c->device = device;
  c->sm_count = prop.multiProcessorCount;
  APS_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
  c->own_stream = true;
  cudaMemPool_t pool;
  APS_CUDA(cudaDeviceGetDefaultMemPool(&pool, device));
  uint64_t thr = UINT64_MAX;
  APS_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr));
  APS_CUDA(cudaMalloc((void**)&c->d_scratch_flags, 64 * sizeof(int32_t)));
  APS_CUDA(cudaMallocHost((void**)&c->h_flags, 64 * sizeof(int32_t)));
  *out = c;
  return APS_OK;
}

extern "C" void aps_ctx_destroy(aps_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  for (cudaEvent_t e : c->tc_events) cudaEventDestroy(e);
  if (c->d_scratch_flags) cudaFree(c->d_scratch_flags);
  if (c->h_flags) cudaFreeHost(c->h_flags);
  if (c->h_stage) cudaFreeHost(c->h_stage);
  if (c->own_stream) cudaStreamDestroy(c->stream);
  delete c;
}

extern "C" int aps_ctx_set_stream(aps_ctx* c, void* cuda_stream) {
  if (!c) APS_FAIL(APS_ERR_ARGS, "", "ctx is NULL");
  APS_CUDA(cudaStreamSynchronize(c->stream));
  if (c->own_stream) cudaStreamDestroy(c->stream);
  c->stream = (cudaStream_t)cuda_stream;
  c->own_stream = false;
  return APS_OK;
}

extern "C" int aps_ctx_synchronize(aps_ctx* c) {
  if (!c) APS_FAIL(APS_ERR_ARGS, "", "ctx is NULL");
  APS_CUDA(cudaStreamSynchronize(c->stream));
  return APS_OK;
}

extern "C" int aps_ctx_enable_timing(aps_ctx* c, int enable) {
  if (!c) APS_FAIL(APS_ERR_ARGS, "", "ctx is NULL");
  c->timing = enable != 0;
  return APS_OK;
}

extern "C" int aps_ctx_tc_time(aps_ctx* c, double* ms_total, int64_t* launches) {
  if (!c || !ms_total || !launches) APS_FAIL(APS_ERR_ARGS, "", "bad args");
  APS_CUDA(cudaSetDevice(c->device));
  APS_CUDA(cudaStreamSynchronize(c->stream));
  double total = 0.0;
  for (size_t i = 0; i + 1 < c->tc_events.size(); i += 2) {
    float ms = 0.f;
    APS_CUDA(cudaEventElapsedTime(&ms, c->tc_events[i], c->tc_events[i + 1]));
    total += ms;
  }
  *ms_total = total;
  *launches = (int64_t)(c->tc_events.size() / 2);
  for (cudaEvent_t e : c->tc_events) cudaEventDestroy(e);
  c->tc_events.clear();
  return APS_OK;
}

extern "C" int aps_ctx_set_float_engine(aps_ctx* c, int engine) {
  if (!c || engine < 0 || engine > 2) APS_FAIL(APS_ERR_ARGS, "", "bad engine");
  c->float_engine = engine;
  return APS_OK;
}
extern "C" int aps_ctx_set_pairwise_epilogue(aps_ctx* c, int mode) {
  if (!c || mode < -1 || mode > 1)
    APS_FAIL(APS_ERR_ARGS, "", "pairwise epilogue must be -1 (auto), 0 (streaming) or 1 (segment selection)");
  c->pairwise_epilogue = mode;
  return APS_OK;
}

extern "C" int aps_ctx_set_pairwise_screen(aps_ctx* c, int mode) {
  if (!c || mode < 0 || mode > 1) APS_FAIL(APS_ERR_ARGS, "", "pairwise screen must be 0 (off) or 1 (on)");
  c->pairwise_screen = mode;
  return APS_OK;
}
extern "C" int aps_ctx_pairwise_stats(aps_ctx* c, int64_t stats[4]) {
  if (!c || !stats) APS_FAIL(APS_ERR_ARGS, "", "bad args");
  for (int i = 0; i < 4; ++i) stats[i] = c->pair_stats[i];
  return APS_OK;
}

extern "C" int64_t aps_ctx_first_pass_unproven(aps_ctx* c) {
  if (!c) return -1;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  return c->h_flags[34];
}

extern "C" int aps_ctx_last_stats(aps_ctx* c, int64_t stats[4]) {
  if (!c || !stats) APS_FAIL(APS_ERR_ARGS, "", "bad args");
  APS_CUDA(cudaSetDevice(c->device));
  APS_CUDA(cudaStreamSynchronize(c->stream));
  if (c->stats[2] == 2) c->stats[1] = c->h_flags[32];  // fallback-row count of the last tensor search
  if (c->h_flags[36] == 1) c->stats[3] = c->h_flags[35] != 0;  // "operands exact in bf16" flag of the last global search
  for (int i = 0; i < 4; ++i) stats[i] = c->stats[i];
  return APS_OK;
}

extern "C" void* aps_host_alloc(size_t bytes) {
  void* p = nullptr;
  if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) return nullptr;
  return p;
}
extern "C" void aps_host_free(void* p) {
  if (p) cudaFreeHost(p);
}


// ------------------------------------------------------------------------------------------------
// staging helpers
int stage_matrix(aps_ctx* c, const void* host, int64_t N, int D, int esz, int layout, void* dst_rm,
                        DevBuf<uint8_t>& tmp) {
  if (N == 0 || D == 0) return APS_OK;
  size_t bytes = (size_t)N * D * esz;
  if (layout == APS_ROW_MAJOR) {
    APS_CUDA(cudaMemcpyAsync(dst_rm, host, bytes, cudaMemcpyHostToDevice, c->stream));
  } else {
    APS_TRY(tmp.alloc(bytes, c->stream));
    APS_CUDA(cudaMemcpyAsync(tmp.p, host, bytes, cudaMemcpyHostToDevice, c->stream));
    APS_TRY(aps_k_transpose_in(c->stream, tmp.p, N, D, esz, dst_rm));
  }
  return APS_OK;
}

__global__ void k_pad_rows_u8(const uint8_t* __restrict__ src, int64_t N, int nb, int nb16, uint8_t* __restrict__ dst) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N * nb16) return;
  int64_t r = i / nb16;
  int c = (int)(i - r * nb16);
  dst[i] = c < nb ? src[r * nb + c] : (uint8_t)0;
}
int pad_rows(cudaStream_t s, const uint8_t* src, int64_t N, int nb, int nb16, uint8_t* dst) {
  if (N == 0) return APS_OK;
  k_pad_rows_u8<<<(unsigned)aps_ceil_div(N * nb16, 256), 256, 0, s>>>(src, N, nb, nb16, dst);
  APS_LAUNCHED();
  return APS_OK;
}


int copy_out_matrix(aps_ctx* c, const uint32_t* idx_rm, const float* dist_rm, int64_t N, int k, int layout,
                           uint32_t* h_idx, float* h_dist) {
  if (N == 0) return APS_OK;
  if (layout == APS_ROW_MAJOR) {
    APS_CUDA(cudaMemcpyAsync(h_idx, idx_rm, (size_t)N * k * 4, cudaMemcpyDeviceToHost, c->stream));
    APS_CUDA(cudaMemcpyAsync(h_dist, dist_rm, (size_t)N * k * 4, cudaMemcpyDeviceToHost, c->stream));
  } else {
    DevBuf<uint32_t> ic;
    DevBuf<float> dc;
    APS_TRY(ic.alloc((size_t)N * k, c->stream));
    APS_TRY(dc.alloc((size_t)N * k, c->stream));
    APS_TRY(aps_k_transpose_out_u32f32(c->stream, idx_rm, dist_rm, N, k, ic.p, dc.p));
    APS_CUDA(cudaMemcpyAsync(h_idx, ic.p, (size_t)N * k * 4, cudaMemcpyDeviceToHost, c->stream));
    APS_CUDA(cudaMemcpyAsync(h_dist, dc.p, (size_t)N * k * 4, cudaMemcpyDeviceToHost, c->stream));
    APS_CUDA(cudaStreamSynchronize(c->stream));
    return APS_OK;
  }
  APS_CUDA(cudaStreamSynchronize(c->stream));
  return APS_OK;
}

// ------------------------------------------------------------------------------------------------
// float search driver: tcgen05 candidates + exact re-rank (+ exact fallback rows), or exact only.

// The completeness proof needs the K'-th candidate strictly beyond the k-th neighbour.  Candidates per list of the tensor
// pass: 8 for k <= 5 (6 when the operands are exact), 16 for 6 <= k <= kTcMaxK -- at least 3 ranks between the k-th
// neighbour and the list's floor.  Larger k stays on the exact engine.
constexpr int kTcMaxK = 12;
static int tc_list_length(int k) { return k <= 5 ? 8 : 16; }

bool tc_wanted(const aps_ctx* c, int D, int64_t nq, int64_t nt, int k) {
  if (c->float_engine == 1) return false;
  if (k > kTcMaxK) return false;
  int Dp = (D + 63) / 64 * 64;
  if (!aps_k_knn_tc_supported(Dp)) return false;
  if (c->float_engine == 2) return true;
  return nq * nt >= (int64_t)1 << 22;  // tiny problems: launch-bound either way, stay exact
}

// Rows the first proof left open: a SHORT list goes straight to the exact engine (its train range is split over 32
// CTAs per 8 rows, aps_knn_exact.cu) -- a second tensor pass over a handful of rows keeps only 4 CTAs busy for a whole
// sweep; a LONG list (real-valued descriptors with tightly packed neighbours) takes the 4-segment tensor pass.
__global__ void k_route_unproven(int32_t* __restrict__ fb, int32_t* __restrict__ n1, int32_t* __restrict__ fb2,
                                 int32_t* __restrict__ n2, int short_list, int32_t* __restrict__ report) {
  __shared__ int n;
  if (threadIdx.x == 0) {
    n = *n1;
    *report = n;
  }
  __syncthreads();
  if (n > short_list) return;
  for (int i = threadIdx.x; i < n; i += blockDim.x) fb2[i] = fb[i];
  __syncthreads();
  if (threadIdx.x == 0) {
    *n2 = n;
    *n1 = 0;
  }
}

// metric 0: FLANN-order squared L2 (global path) ; metric 1: SSD (pairwise path)
int float_knn(aps_ctx* c, const FloatSide& Q, int64_t q0, int64_t q1, const FloatSide& T, int64_t t0,
                     int64_t t1, int D, int k, int metric, int bias_mode, const int32_t* flags_dev,
                     int64_t out_row0, uint32_t* idx, float* dist, bool use_tc) {
  const int64_t nq = q1 - q0;
  if (nq <= 0) return APS_OK;
  c->stats[0] += nq;
  if (!use_tc || t1 - t0 < k + 1) {
    c->stats[2] = 1;
    return aps_k_knn_exact(c->stream, Q.xn, Q.sq, nullptr, nullptr, q0, nq, T.xn, T.sq, t0, t1, D, k, metric,
                           out_row0, idx, dist);
  }
  c->stats[2] = 2;
  const int Dp = (D + 63) / 64 * 64;
  const int kcand = tc_list_length(k);
  const int kcap_exact = kcand == 8 ? 6 : 0;  // K' = 16 has no exact-operand variant
  const int nslot = aps_k_knn_tc_slots(c->sm_count, nq, t0, t1);  // candidate lists per row (tail balancing)
  DevBuf<uint32_t> cidx;
  DevBuf<float> cscore;
  DevBuf<int32_t> fb;
  APS_TRY(cidx.alloc((size_t)nq * nslot * kcand, c->stream));
  APS_TRY(cscore.alloc((size_t)nq * nslot * kcand, c->stream));
  APS_TRY(fb.alloc((size_t)nq + 1, c->stream));
  APS_CUDA(cudaMemsetAsync(fb.p + nq, 0, sizeof(int32_t), c->stream));
  aps_tc_problem p;
  p.Qb = Q.xb;
  p.Tb = T.xb_t;
  p.colscale = T.colscale_t;
  p.colbias = T.colbias_t;
  p.tile_bounds = T.tile_bounds;
  p.bias = bias_mode;
  p.Fq_total = Q.N;
  p.Ft_total = T.N;
  p.Dp = Dp;
  p.q0 = q0;
  p.q1 = q1;
  p.t0 = t0;
  p.t1 = t1;
  p.nslot = nslot;
  p.kcand = kcand;
  p.cand_idx = cidx.p;
  p.cand_score = cscore.p;
  p.dump = nullptr;
  p.operand_fp16 = (Q.fp16 && T.fp16) ? 2 : 0;
  aps_pair_tables gpt;       // global searches: only the operand kind travels in here (eoff == nullptr)
  memset(&gpt, 0, sizeof gpt);
  gpt.operand_fp16 = p.operand_fp16;
  p.exact_flag = flags_dev;  // exact operands (integer SIFT): 6 candidates per list are enough to prove a top-5 (K' = 8)
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  if (c->timing) {
    APS_CUDA(cudaEventCreate(&ev0));
    APS_CUDA(cudaEventCreate(&ev1));
  }
  APS_TRY(aps_k_knn_tc(c->stream, c->sm_count, p, ev0, ev1));
  if (c->timing) {
    c->tc_events.push_back(ev0);
    c->tc_events.push_back(ev1);
  }
  // rows of full-width units keep all their candidates in list 0: kcand lanes per row instead of nslot * kcand
  const int64_t rows_full = nslot > 1 ? aps_k_knn_tc_full_rows(c->sm_count, nq, t0, t1) : 0;
  if (rows_full > 0)
    APS_TRY(aps_k_rerank(c->stream, Q.xn, Q.sq, Q.invn, T.xn, T.sq, D, metric, q0, rows_full, t0, 1, kcand, cidx.p,
                         cscore.p, flags_dev, bias_mode, flags_dev, k, out_row0, idx, dist, fb.p, fb.p + nq, &gpt,
                         nullptr, nullptr, T.perm, nslot * kcand, kcap_exact));
  if (nq > rows_full)
    APS_TRY(aps_k_rerank(c->stream, Q.xn, Q.sq, Q.invn, T.xn, T.sq, D, metric, q0 + rows_full, nq - rows_full, t0, nslot,
                         kcand, cidx.p + (size_t)rows_full * nslot * kcand, cscore.p + (size_t)rows_full * nslot * kcand,
                         flags_dev, bias_mode, flags_dev, k, out_row0, idx, dist, fb.p, fb.p + nq, &gpt, nullptr,
                         nullptr, T.perm, 0, kcap_exact));
  // Rows that could not be proven complete (device-side list, no host round trip) get a SECOND tensor pass with
  // 4 column segments = 4 * kcand (32 or 64) candidates per row: with inexact (non bf16-representable) operands the error
  // bound is ~0.016 in squared distance and 8 candidates often do not reach beyond it; 32 usually do.
  const int nslot2 = aps_k_knn_tc_slots(c->sm_count, nq, t0, t1, /*all_segmented*/ 1);
  DevBuf<int32_t> fb2;
  APS_TRY(fb2.alloc((size_t)nq + 1, c->stream));
  APS_CUDA(cudaMemsetAsync(fb2.p + nq, 0, sizeof(int32_t), c->stream));
  if (nslot2 > nslot) {
    k_route_unproven<<<1, 256, 0, c->stream>>>(fb.p, fb.p + nq, fb2.p, fb2.p + nq, /*short_list*/ 128,
                                               c->d_scratch_flags + 8);
    APS_LAUNCHED();
    APS_CUDA(cudaMemcpyAsync(c->h_flags + 34, c->d_scratch_flags + 8, sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
    DevBuf<__nv_bfloat16> qb2;
    DevBuf<uint32_t> cidx2;
    DevBuf<float> cscore2;
    APS_TRY(qb2.alloc((size_t)nq * Dp, c->stream));
    APS_TRY(cidx2.alloc((size_t)nq * nslot2 * kcand, c->stream));
    APS_TRY(cscore2.alloc((size_t)nq * nslot2 * kcand, c->stream));
    APS_TRY(aps_k_gather_rows(c->stream, Q.xb, Dp, fb.p, fb.p + nq, nq, qb2.p));
    aps_tc_problem p2 = p;
    p2.Qb = qb2.p;
    p2.Fq_total = nq;
    p2.q0 = 0;
    p2.q1 = nq;
    p2.nslot = nslot2;
    p2.cand_idx = cidx2.p;
    p2.cand_score = cscore2.p;
    p2.nrows_dev = fb.p + nq;
    APS_TRY(aps_k_knn_tc(c->stream, c->sm_count, p2, nullptr, nullptr));
    APS_TRY(aps_k_rerank(c->stream, Q.xn, Q.sq, Q.invn, T.xn, T.sq, D, metric, q0, nq, t0, nslot2, kcand, cidx2.p,
                         cscore2.p, flags_dev, bias_mode, flags_dev, k, out_row0, idx, dist, fb2.p, fb2.p + nq, &gpt,
                         fb.p, fb.p + nq, T.perm));
    // still unproven: exact CUDA-core search
    APS_TRY(aps_k_knn_exact(c->stream, Q.xn, Q.sq, fb2.p, fb2.p + nq, q0, nq, T.xn, T.sq, t0, t1, D, k, metric,
                            out_row0, idx, dist));
    APS_CUDA(cudaMemcpyAsync(c->h_flags + 32, fb2.p + nq, sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
  } else {
    APS_TRY(aps_k_knn_exact(c->stream, Q.xn, Q.sq, fb.p, fb.p + nq, q0, nq, T.xn, T.sq, t0, t1, D, k, metric,
                            out_row0, idx, dist));
    APS_CUDA(cudaMemcpyAsync(c->h_flags + 32, fb.p + nq, sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
    APS_CUDA(cudaMemcpyAsync(c->h_flags + 34, fb.p + nq, sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
  }
  return APS_OK;
}


int floatset_alloc(aps_ctx* c, FloatSet& fs, int64_t N, int D) {
  fs.N = N;
  fs.D = D;
  APS_TRY(fs.raw.alloc((size_t)N * D, c->stream));
  APS_TRY(fs.sq.alloc((size_t)N, c->stream));
  APS_TRY(fs.invn.alloc((size_t)N, c->stream));
  APS_TRY(fs.flags.alloc(8, c->stream));
  return APS_OK;
}

int floatset_reset_flags(aps_ctx* c, FloatSet& fs) {
  static const int32_t init[8] = {1, 0, 0, 0, 0, 0, 0, 0};
  APS_CUDA(cudaMemcpyAsync(fs.flags.p, init, sizeof init, cudaMemcpyHostToDevice, c->stream));
  return APS_OK;
}

// Train-side view of the tensor kernel: rows bucket-sorted by scale when `sort` (whole-set searches; pairwise
// units need each image's rows contiguous and keep the natural order) + per-tile pre-filter bounds.
int floatset_finish_train(aps_ctx* c, FloatSet& fs, bool sort) {
  if (fs.N == 0 || !fs.xb.p) return APS_OK;
  const int Dp = (fs.D + 63) / 64 * 64;
  fs.sorted = false;
  if (sort) {
    APS_TRY(fs.xb_t.alloc((size_t)fs.N * Dp, c->stream));
    APS_TRY(fs.colscale_t.alloc((size_t)fs.N + 256, c->stream));
    APS_TRY(fs.colbias_t.alloc((size_t)fs.N + 256, c->stream));
    APS_TRY(fs.perm.alloc((size_t)fs.N, c->stream));
    APS_TRY(fs.sort_scratch.alloc((size_t)aps_sort_scratch_ints(), c->stream));
    APS_TRY(aps_k_sort_train_by_scale(c->stream, fs.xb.p, fs.colscale.p, fs.colbias.p, fs.N, Dp, fs.sort_scratch.p,
                                      fs.perm.p, fs.xb_t.p, fs.colscale_t.p, fs.colbias_t.p));
    fs.sorted = true;
  }
  const int tr = aps_k_knn_tc_tile_rows();
  APS_TRY(fs.tile_bounds.alloc((size_t)aps_ceil_div(fs.N, tr) + 2, c->stream));
  APS_TRY(aps_k_tile_bounds(c->stream, fs.sorted ? fs.colscale_t.p : fs.colscale.p,
                            fs.sorted ? fs.colbias_t.p : fs.colbias.p, fs.N, tr, fs.tile_bounds.p));
  return APS_OK;
}

// normalise + (optionally) build tensor operands
int floatset_prepare(aps_ctx* c, FloatSet& fs, int norm_mode, bool tensor, int bias_mode, bool sort) {
  if (fs.N == 0) return APS_OK;
  if (norm_mode != APS_NORM_NONE && !fs.xn.p) APS_TRY(fs.xn.alloc((size_t)fs.N * fs.D, c->stream));
  float* xn = (norm_mode != APS_NORM_NONE) ? fs.xn.p : fs.raw.p;
  APS_TRY(aps_k_prepare_norm(c->stream, fs.raw.p, fs.N, fs.D, norm_mode, xn, fs.sq.p, fs.invn.p, fs.flags.p, fs.fp16));
  if (tensor) {
    const int Dp = (fs.D + 63) / 64 * 64;
    APS_TRY(fs.xb.alloc((size_t)fs.N * Dp, c->stream));
    APS_TRY(fs.colscale.alloc((size_t)fs.N + 256, c->stream));
    APS_TRY(fs.colbias.alloc((size_t)fs.N + 256, c->stream));  // +256: whole-tile bulk loads
    APS_TRY(aps_k_prepare_operands(c->stream, fs.raw.p, xn, fs.sq.p, fs.invn.p, fs.N, fs.D, Dp, fs.flags.p,
                                   bias_mode, fs.xb.p, fs.colscale.p, fs.colbias.p, fs.fp16));
    APS_TRY(floatset_finish_train(c, fs, sort));
  }
  return APS_OK;
}

// ------------------------------------------------------------------------------------------------
// flann_knn_win
extern "C" int aps_flann_knn(aps_ctx* c, const void* train, int64_t Ft, const void* query, int64_t Fq, int D,
                             int dtype, int layout, int k, const char* method, int trees, int checks,
                             uint32_t* idx, float* dist) {
  (void)trees;
  (void)checks;
  APS_CTX(c);
  if (dtype != APS_F32 && dtype != APS_U8)
    APS_FAIL(APS_ERR_TYPE, "flann_knn:type", "Descriptors must be single (float) or uint8 (binary)");
  if (k <= 0) APS_FAIL(APS_ERR_K, "flann_knn:k", "k must be > 0");
  if (k > APS_MAX_K) APS_FAIL(APS_ERR_K, "flann_knn:k", "k must be <= %d in this implementation", APS_MAX_K);
  if (D <= 0 && (Ft > 0 || Fq > 0)) APS_FAIL(APS_ERR_DIM, "flann_knn:dim", "descriptor dimension must be positive");
  std::string m = method ? method : "flann";
  if (m != "flann" && m != "bf") APS_FAIL(APS_ERR_METHOD, "flann_knn:args", "unknown method '%s'", m.c_str());
  if (m == "bf" && dtype != APS_U8)
    APS_FAIL(APS_ERR_BF, "flann_knn:bf", "BFMatcher only supports uint8 (binary) descriptors");
  if ((Ft > 0 && !train) || (Fq > 0 && (!query || !idx || !dist)))
    APS_FAIL(APS_ERR_ARGS, "flann_knn:args", "null pointer argument");
  if (Fq == 0) return APS_OK;
  c->stats[0] = c->stats[1] = c->stats[2] = c->stats[3] = 0;
  DevBuf<uint32_t> didx;
  DevBuf<float> ddist;
  DevBuf<uint8_t> tmp;
  APS_TRY(didx.alloc((size_t)Fq * k, c->stream));
  APS_TRY(ddist.alloc((size_t)Fq * k, c->stream));
  const bool self = (train == query && Ft == Fq);
  if (dtype == APS_U8) {
    const int nb16 = (D + 15) / 16 * 16;
    DevBuf<uint8_t> t_raw, q_raw, t_pad, q_pad;
    APS_TRY(t_raw.alloc((size_t)Ft * D, c->stream));
    APS_TRY(t_pad.alloc((size_t)Ft * nb16, c->stream));
    APS_TRY(stage_matrix(c, train, Ft, D, 1, layout, t_raw.p, tmp));
    APS_TRY(pad_rows(c->stream, t_raw.p, Ft, D, nb16, t_pad.p));
    const uint8_t* qp = t_pad.p;
    if (!self) {
      APS_TRY(q_raw.alloc((size_t)Fq * D, c->stream));
      APS_TRY(q_pad.alloc((size_t)Fq * nb16, c->stream));
      APS_TRY(stage_matrix(c, query, Fq, D, 1, layout, q_raw.p, tmp));
      APS_TRY(pad_rows(c->stream, q_raw.p, Fq, D, nb16, q_pad.p));
      qp = q_pad.p;
    }
    APS_TRY(aps_k_knn_hamming(c->stream, qp, 0, Fq, t_pad.p, 0, Ft, nb16, k, 0, didx.p, ddist.p));
    c->stats[0] = Fq;
    c->stats[2] = 1;
    return copy_out_matrix(c, didx.p, ddist.p, Fq, k, layout, idx, dist);
  }
  // float: the caller passes what featureMatchingGlobal.m:80-84 already normalised -> no normalisation here
  const bool tc = tc_wanted(c, D, Fq, Ft, k);
  FloatSet T, Q;
  APS_TRY(floatset_alloc(c, T, Ft, D));
  APS_TRY(floatset_reset_flags(c, T));
  APS_TRY(stage_matrix(c, train, Ft, D, 4, layout, T.raw.p, tmp));
  APS_TRY(floatset_prepare(c, T, APS_NORM_NONE, tc, /*bias: rows need not be unit norm*/ 1));
  FloatSide qs = T.side();
  if (!self) {
    APS_TRY(floatset_alloc(c, Q, Fq, D));
    Q.flags.release();
    // share the flag words with the train set: exactness / magnitude bounds must hold for both sides
    APS_TRY(stage_matrix(c, query, Fq, D, 4, layout, Q.raw.p, tmp));
    if (Fq > 0) {
      APS_TRY(aps_k_prepare_norm(c->stream, Q.raw.p, Fq, D, APS_NORM_NONE, Q.raw.p, Q.sq.p, Q.invn.p, T.flags.p));
      if (tc) {
        const int Dp = (D + 63) / 64 * 64;
        APS_TRY(Q.xb.alloc((size_t)Fq * Dp, c->stream));
        APS_TRY(Q.colscale.alloc((size_t)Fq + 256, c->stream));
    APS_TRY(Q.colbias.alloc((size_t)Fq + 256, c->stream));
        // NOTE: operands of BOTH sides are built after both flag passes ran (same stream order)
        APS_TRY(aps_k_prepare_operands(c->stream, Q.raw.p, Q.raw.p, Q.sq.p, Q.invn.p, Fq, D, Dp, T.flags.p, 1,
                                       Q.xb.p, Q.colscale.p, Q.colbias.p));
        APS_TRY(aps_k_prepare_operands(c->stream, T.raw.p, T.raw.p, T.sq.p, T.invn.p, Ft, D, Dp, T.flags.p, 1,
                                       T.xb.p, T.colscale.p, T.colbias.p));
        APS_TRY(floatset_finish_train(c, T, true));
      }
    }
    qs = Q.side();
    qs.xn = Q.raw.p;
  }
  APS_TRY(float_knn(c, qs, 0, Fq, T.side(), 0, Ft, D, k, /*metric*/ 0, /*bias_mode*/ 1, T.flags.p, 0, didx.p,
                    ddist.p, tc));
  int rc = copy_out_matrix(c, didx.p, ddist.p, Fq, k, layout, idx, dist);
  c->stats[1] = c->h_flags[32];
  return rc;
}

// ------------------------------------------------------------------------------------------------
// nearest2HammingExhaustive{,OMP}MEX
int hamming2_device(aps_ctx* c, const uint8_t* qpad, int64_t q0, int64_t N1, const uint8_t* tpad, int64_t t0,
                           int64_t N2, int nb, int nb16, uint32_t* idx2, float* d1, float* d2) {
  DevBuf<uint32_t> i2;
  DevBuf<float> dd;
  APS_TRY(i2.alloc((size_t)N1 * 2, c->stream));
  APS_TRY(dd.alloc((size_t)N1 * 2, c->stream));
  if (N2 > 0) APS_TRY(aps_k_knn_hamming(c->stream, qpad, q0, N1, tpad, t0, t0 + N2, nb16, 2, q0, i2.p, dd.p));
  APS_TRY(aps_k_hamming2_finalize(c->stream, N1, N2, nb, i2.p, dd.p, idx2, d1, d2));
  return APS_OK;
}

extern "C" int aps_nearest2_hamming(aps_ctx* c, const uint8_t* A, int64_t N1, const uint8_t* B, int64_t N2, int nb,
                                    int layout, uint32_t* idx2, float* d1, float* d2) {
  APS_CTX(c);
  if ((N1 > 0 && (!A || !idx2 || !d1 || !d2)) || (N2 > 0 && !B))
    APS_FAIL(APS_ERR_ARGS, "hamm2nn:nrhs", "Need Abytes,Bbytes");
  if (nb <= 0 && (N1 > 0 || N2 > 0)) APS_FAIL(APS_ERR_DIM, "hamm2nn:cols", "Byte width mismatch.");
  if (N1 == 0) return APS_OK;
  const int nb16 = (nb + 15) / 16 * 16;
  DevBuf<uint8_t> a_raw, b_raw, a_pad, b_pad, tmp;
  APS_TRY(a_raw.alloc((size_t)N1 * nb, c->stream));
  APS_TRY(a_pad.alloc((size_t)N1 * nb16, c->stream));
  APS_TRY(b_raw.alloc((size_t)N2 * nb, c->stream));
  APS_TRY(b_pad.alloc((size_t)N2 * nb16, c->stream));
  APS_TRY(stage_matrix(c, A, N1, nb, 1, layout, a_raw.p, tmp));
  APS_TRY(stage_matrix(c, B, N2, nb, 1, layout, b_raw.p, tmp));
  APS_TRY(pad_rows(c->stream, a_raw.p, N1, nb, nb16, a_pad.p));
  APS_TRY(pad_rows(c->stream, b_raw.p, N2, nb, nb16, b_pad.p));
  DevBuf<uint32_t> di;
  DevBuf<float> dd1, dd2;
  APS_TRY(di.alloc((size_t)N1, c->stream));
  APS_TRY(dd1.alloc((size_t)N1, c->stream));
  APS_TRY(dd2.alloc((size_t)N1, c->stream));
  APS_TRY(hamming2_device(c, a_pad.p, 0, N1, b_pad.p, 0, N2, nb, nb16, di.p, dd1.p, dd2.p));
  APS_CUDA(cudaMemcpyAsync(idx2, di.p, (size_t)N1 * 4, cudaMemcpyDeviceToHost, c->stream));
  APS_CUDA(cudaMemcpyAsync(d1, dd1.p, (size_t)N1 * 4, cudaMemcpyDeviceToHost, c->stream));
  APS_CUDA(cudaMemcpyAsync(d2, dd2.p, (size_t)N1 * 4, cudaMemcpyDeviceToHost, c->stream));
  APS_CUDA(cudaStreamSynchronize(c->stream));
  return APS_OK;
}

// ------------------------------------------------------------------------------------------------
// nearest2SSDExhaustive (device part shared with matchFeaturesScratch / pairwise)
int ssd2_device(aps_ctx* c, const FloatSide& Q, int64_t q0, int64_t N1, const FloatSide& T, int64_t t0,
                       int64_t N2, int D, const int32_t* flags, bool tc, int bias_mode, uint32_t* idx2, float* d1,
                       float* d2) {
  DevBuf<uint32_t> i2;
  DevBuf<float> dd;
  APS_TRY(i2.alloc((size_t)N1 * 2, c->stream));
  APS_TRY(dd.alloc((size_t)N1 * 2, c->stream));
  if (N2 > 0) {
    APS_TRY(float_knn(c, Q, q0, q0 + N1, T, t0, t0 + N2, D, 2, /*metric*/ 1, bias_mode, flags, q0, i2.p, dd.p, tc));
  } else {
    // N2 == 0 -> idx 0, +inf, +inf (documented deviation: MATLAB's validateattributes throws)
    APS_CUDA(cudaMemsetAsync(i2.p, 0, (size_t)N1 * 2 * 4, c->stream));
    std::vector<float> inf((size_t)N1 * 2, std::numeric_limits<float>::infinity());
    APS_CUDA(cudaMemcpyAsync(dd.p, inf.data(), inf.size() * 4, cudaMemcpyHostToDevice, c->stream));
    APS_CUDA(cudaStreamSynchronize(c->stream));
  }
  APS_TRY(aps_k_split_k2(c->stream, N1, i2.p, dd.p, idx2, d1, d2));
  return APS_OK;
}

extern "C" int aps_nearest2_ssd(aps_ctx* c, const float* A, int64_t N1, const float* B, int64_t N2, int D,
                                int layout, uint32_t* idx2, float* d1, float* d2) {
  APS_CTX(c);
  if ((N1 > 0 && (!A || !idx2 || !d1 || !d2)) || (N2 > 0 && !B)) APS_FAIL(APS_ERR_ARGS, "", "null pointer argument");
  if (D <= 0) APS_FAIL(APS_ERR_DIM, "", "descriptor dimension must be positive");
  if (N1 == 0) return APS_OK;
  c->stats[0] = c->stats[1] = c->stats[2] = c->stats[3] = 0;
  const bool tc = tc_wanted(c, D, N1, N2, 2);
  FloatSet QA, TB;
  DevBuf<uint8_t> tmp;
  APS_TRY(floatset_alloc(c, QA, N1, D));
  APS_TRY(floatset_alloc(c, TB, N2, D));
  APS_TRY(floatset_reset_flags(c, TB));
  APS_TRY(stage_matrix(c, A, N1, D, 4, layout, QA.raw.p, tmp));
  APS_TRY(stage_matrix(c, B, N2, D, 4, layout, TB.raw.p, tmp));
  APS_TRY(aps_k_prepare_norm(c->stream, QA.raw.p, N1, D, APS_NORM_NONE, QA.raw.p, QA.sq.p, QA.invn.p, TB.flags.p));
  APS_TRY(aps_k_prepare_norm(c->stream, TB.raw.p, N2, D, APS_NORM_NONE, TB.raw.p, TB.sq.p, TB.invn.p, TB.flags.p));
  if (tc) {
    const int Dp = (D + 63) / 64 * 64;
    APS_TRY(QA.xb.alloc((size_t)N1 * Dp, c->stream));
    APS_TRY(QA.colscale.alloc((size_t)N1 + 256, c->stream));
    APS_TRY(QA.colbias.alloc((size_t)N1 + 256, c->stream));
    APS_TRY(TB.xb.alloc((size_t)N2 * Dp, c->stream));
    APS_TRY(TB.colscale.alloc((size_t)N2 + 256, c->stream));
    APS_TRY(TB.colbias.alloc((size_t)N2 + 256, c->stream));
    APS_TRY(aps_k_prepare_operands(c->stream, QA.raw.p, QA.raw.p, QA.sq.p, QA.invn.p, N1, D, Dp, TB.flags.p, 1,
                                   QA.xb.p, QA.colscale.p, QA.colbias.p));
    APS_TRY(aps_k_prepare_operands(c->stream, TB.raw.p, TB.raw.p, TB.sq.p, TB.invn.p, N2, D, Dp, TB.flags.p, 1,
                                   TB.xb.p, TB.colscale.p, TB.colbias.p));
    APS_TRY(floatset_finish_train(c, TB, true));
  }
  DevBuf<uint32_t> di;
  DevBuf<float> dd1, dd2;
  APS_TRY(di.alloc((size_t)N1, c->stream));
  APS_TRY(dd1.alloc((size_t)N1, c->stream));
  APS_TRY(dd2.alloc((size_t)N1, c->stream));
  APS_TRY(ssd2_device(c, QA.side(), 0, N1, TB.side(), 0, N2, D, TB.flags.p, tc, 1, di.p, dd1.p, dd2.p));
  APS_CUDA(cudaMemcpyAsync(idx2, di.p, (size_t)N1 * 4, cudaMemcpyDeviceToHost, c->stream));
  APS_CUDA(cudaMemcpyAsync(d1, dd1.p, (size_t)N1 * 4, cudaMemcpyDeviceToHost, c->stream));
  APS_CUDA(cudaMemcpyAsync(d2, dd2.p, (size_t)N1 * 4, cudaMemcpyDeviceToHost, c->stream));
  APS_CUDA(cudaStreamSynchronize(c->stream));
  c->stats[1] = c->h_flags[32];
  return APS_OK;
}

// ------------------------------------------------------------------------------------------------
// match lists
extern "C" int aps_matchlist_n(const aps_matchlist* m) { return m ? m->n : 0; }
extern "C" int64_t aps_matchlist_total(const aps_matchlist* m) { return m ? m->total : 0; }
extern "C" const int64_t* aps_matchlist_pair_ptr(const aps_matchlist* m) { return m ? m->pair_ptr.data() : nullptr; }
extern "C" const uint32_t* aps_matchlist_rows(const aps_matchlist* m) { return m ? m->rows.data() : nullptr; }
extern "C" const double* aps_matchlist_metric(const aps_matchlist* m) {
  return (m && m->has_metric) ? m->metric.data() : nullptr;
}
extern "C" void aps_matchlist_free(aps_matchlist* m) { delete m; }

// ------------------------------------------------------------------------------------------------
// staged global pipeline
struct aps_gplan {
  aps_ctx* c = nullptr;
  int n = 0, D = 0, dtype = 0, k = 0;
  int64_t F = 0, maxcount = 0;
  std::vector<int64_t> counts, off;
  bool tensor = false;
  // descriptors
  FloatSet fs;                    // float
  DevBuf<uint8_t> u8raw, u8pad;   // binary
  int nb16 = 0;
  DevBuf<uint8_t> stage_tmp;
  // bookkeeping
  DevBuf<int64_t> d_off;
  DevBuf<int32_t> img_of_row;
  // results
  DevBuf<uint32_t> knn_idx;
  DevBuf<float> knn_dist;
  DevBuf<int2> records;     // [F + APS_RECORD_PAD]: (target image + 1 | 0, partner's local index) per query row; the
                            // padding lets equal-sized rank slices of an in-place all-gather run past F
  DevBuf<int64_t> dir_counts, pair_counts, pair_ptr, rank;
  DevBuf<uint32_t> rows;
  bool compacted = false;
};

extern "C" int aps_gplan_create(aps_ctx* c, const int64_t* counts, int n, int D, int dtype, int k, aps_gplan** out) {
  APS_CTX(c);
  if (!out || n < 0 || (n > 0 && !counts)) APS_FAIL(APS_ERR_ARGS, "", "bad arguments");
  if (dtype != APS_F32 && dtype != APS_U8)
    APS_FAIL(APS_ERR_TYPE, "flann_knn:type", "Descriptors must be single (float) or uint8 (binary)");
  if (k <= 0) APS_FAIL(APS_ERR_K, "flann_knn:k", "k must be > 0");
  if (k > APS_MAX_K) APS_FAIL(APS_ERR_K, "flann_knn:k", "k must be <= %d in this implementation", APS_MAX_K);
  aps_gplan* p = new (std::nothrow) aps_gplan();
  if (!p) APS_FAIL(APS_ERR_ALLOC, "", "out of host memory");
  p->c = c;
  p->n = n;
  p->D = D;
  p->dtype = dtype;
  p->k = k;
  p->counts.assign(counts, counts + n);
  p->off.assign(n + 1, 0);
  for (int i = 0; i < n; ++i) {
    if (counts[i] < 0) {
      delete p;
      APS_FAIL(APS_ERR_ARGS, "", "negative feature count");
    }
    p->off[i + 1] = p->off[i] + counts[i];
    if (counts[i] > p->maxcount) p->maxcount = counts[i];
  }
  p->F = p->off[n];
  if (p->F > 0 && D <= 0) {
    delete p;
    APS_FAIL(APS_ERR_DIM, "flann_knn:dim", "descriptor dimension must be positive");
  }
  if (p->F >= ((int64_t)1 << 31) - 1) {
    delete p;
    APS_FAIL(APS_ERR_ARGS, "", "more than 2^31 descriptors are not supported");
  }
  const int64_t F = p->F;
  cudaStream_t s = c->stream;
  int rc = APS_OK;
  auto A = [&](int r) { if (rc == APS_OK) rc = r; };
  if (dtype == APS_F32) {
    p->tensor = tc_wanted(c, D, F, F, k);
    p->fs.fp16 = true;  // rows are L2-normalised (|x| <= 1) or, when exact, small integers: always inside the fp16 range
    A(floatset_alloc(c, p->fs, F, D));
  } else {
    p->nb16 = (D + 15) / 16 * 16;
    A(p->u8raw.alloc((size_t)F * D, s));
    A(p->u8pad.alloc((size_t)F * p->nb16, s));
  }
  A(p->d_off.alloc((size_t)n + 1, s));
  A(p->img_of_row.alloc((size_t)F, s));
  A(p->knn_idx.alloc((size_t)F * k, s));
  A(p->knn_dist.alloc((size_t)F * k, s));
  A(p->records.alloc((size_t)F + APS_RECORD_PAD, s));
  A(p->dir_counts.alloc((size_t)n * n, s));
  A(p->pair_counts.alloc((size_t)n * n, s));
  A(p->pair_ptr.alloc((size_t)n * n + 1, s));
  A(p->rank.alloc((size_t)F, s));
  A(p->rows.alloc((size_t)F * 2, s));
  if (rc == APS_OK && cudaMemcpyAsync(p->d_off.p, p->off.data(), (size_t)(n + 1) * 8, cudaMemcpyHostToDevice, s) != cudaSuccess)
    rc = APS_ERR_CUDA;
  if (rc == APS_OK) rc = aps_k_fill_img_of_row(s, p->d_off.p, n, p->maxcount, p->img_of_row.p);
  if (rc == APS_OK && F > 0 && cudaMemsetAsync(p->records.p, 0, ((size_t)F + APS_RECORD_PAD) * 8, s) != cudaSuccess) rc = APS_ERR_CUDA;
  if (rc != APS_OK) {
    delete p;
    return rc;
  }
  *out = p;
  return APS_OK;
}

extern "C" void aps_gplan_destroy(aps_gplan* p) {
  if (!p) return;
  cudaSetDevice(p->c->device);
  delete p;
}
extern "C" int64_t aps_gplan_total(const aps_gplan* p) { return p ? p->F : 0; }
extern "C" void* aps_gplan_desc_device(aps_gplan* p) {
  if (!p) return nullptr;
  return p->dtype == APS_F32 ? (void*)p->fs.raw.p : (void*)p->u8raw.p;
}
extern "C" void* aps_gplan_records_device(aps_gplan* p) { return p ? p->records.p : nullptr; }
extern "C" void* aps_gplan_knn_idx_device(aps_gplan* p) { return p ? p->knn_idx.p : nullptr; }
extern "C" void* aps_gplan_knn_dist_device(aps_gplan* p) { return p ? p->knn_dist.p : nullptr; }

extern "C" int aps_gplan_upload(aps_gplan* p, const void* const* desc, int layout) {
  return gplan_upload_images(p, desc, layout, 0, p ? p->n : 0);
}

// H2D of images [i0, i1) only, into their rows of the pooled matrix (a device group's members each upload one range)
int gplan_upload_images(aps_gplan* p, const void* const* desc, int layout, int i0, int i1) {
  if (!p) APS_FAIL(APS_ERR_ARGS, "", "plan is NULL");
  aps_ctx* c = p->c;
  APS_CTX(c);
  if (i0 < 0 || i1 > p->n || i0 > i1) APS_FAIL(APS_ERR_ARGS, "", "image range out of bounds");
  const int esz = p->dtype == APS_F32 ? 4 : 1;
  char* base = (char*)aps_gplan_desc_device(p);
  const int64_t r0 = p->off[i0], rows = p->off[i1] - r0;
  if (layout == APS_COL_MAJOR && rows > 0) APS_TRY(p->stage_tmp.alloc((size_t)rows * p->D * esz, c->stream));
  for (int i = i0; i < i1; ++i) {
    const int64_t Ni = p->counts[i];
    if (Ni == 0) continue;
    if (!desc || !desc[i]) APS_FAIL(APS_ERR_ARGS, "", "descriptor pointer %d is NULL but its count is %lld", i, (long long)Ni);
    char* dst = base + (size_t)p->off[i] * p->D * esz;
    size_t bytes = (size_t)Ni * p->D * esz;
    if (layout == APS_ROW_MAJOR) {
      APS_CUDA(cudaMemcpyAsync(dst, desc[i], bytes, cudaMemcpyHostToDevice, c->stream));
    } else {
      char* st = (char*)p->stage_tmp.p + (size_t)(p->off[i] - r0) * p->D * esz;
      APS_CUDA(cudaMemcpyAsync(st, desc[i], bytes, cudaMemcpyHostToDevice, c->stream));
      APS_TRY(aps_k_transpose_in(c->stream, st, Ni, p->D, esz, dst));
    }
  }
  return APS_OK;
}

extern "C" int aps_gplan_prepare(aps_gplan* p) {
  if (!p) APS_FAIL(APS_ERR_ARGS, "", "plan is NULL");
  aps_ctx* c = p->c;
  APS_CTX(c);
  if (p->F == 0) return APS_OK;
  if (p->dtype == APS_F32) {
    APS_TRY(floatset_reset_flags(c, p->fs));
    // featureMatchingGlobal.m:80-84 ; operands: scale-only scoring (rows are unit norm up to rounding)
    APS_TRY(floatset_prepare(c, p->fs, APS_NORM_GLOBAL, p->tensor, /*bias_mode*/ 0));
  } else {
    APS_TRY(pad_rows(c->stream, p->u8raw.p, p->F, p->D, p->nb16, p->u8pad.p));
  }
  return APS_OK;
}

extern "C" int aps_gplan_knn(aps_gplan* p, int64_t q0, int64_t q1) {
  if (!p) APS_FAIL(APS_ERR_ARGS, "", "plan is NULL");
  aps_ctx* c = p->c;
  APS_CTX(c);
  if (q0 < 0 || q1 > p->F || q0 > q1) APS_FAIL(APS_ERR_ARGS, "", "query range out of bounds");
  c->stats[0] = c->stats[1] = c->stats[2] = c->stats[3] = 0;  // an empty range reports an empty search
  c->h_flags[36] = 0;
  if (q0 == q1) return APS_OK;
  if (p->dtype == APS_F32) {
    FloatSide s = p->fs.side();
    APS_TRY(float_knn(c, s, q0, q1, s, 0, p->F, p->D, p->k, /*metric*/ 0, /*bias*/ 0, p->fs.flags.p, 0,
                      p->knn_idx.p, p->knn_dist.p, p->tensor));
    APS_CUDA(cudaMemcpyAsync(c->h_flags + 35, p->fs.flags.p, sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
    c->h_flags[36] = 1;
  } else {
    APS_TRY(aps_k_knn_hamming(c->stream, p->u8pad.p, q0, q1 - q0, p->u8pad.p, 0, p->F, p->nb16, p->k, 0,
                              p->knn_idx.p, p->knn_dist.p));
    c->stats[0] = q1 - q0;
    c->stats[2] = 1;
  }
  return APS_OK;
}

extern "C" int aps_gplan_filter(aps_gplan* p, int64_t q0, int64_t q1, double ratio) {
  if (!p) APS_FAIL(APS_ERR_ARGS, "", "plan is NULL");
  aps_ctx* c = p->c;
  APS_CTX(c);
  if (q0 < 0 || q1 > p->F || q0 > q1) APS_FAIL(APS_ERR_ARGS, "", "query range out of bounds");
  return aps_k_global_filter(c->stream, p->knn_idx.p, p->knn_dist.p, p->k, q0, q1, p->img_of_row.p, p->d_off.p,
                             (float)ratio, p->records.p);
}

// Opt-in cross-check on the GLOBAL path (off in the reference: featureMatchingGlobal.m:149-159 keeps A->B and B->A rows
// alike, BFMatcher is built with crossCheck = false, flann_knn.cpp:204).  Runs on the complete record set (after the
// ranks exchanged their slices): a query keeps its match only if the matched feature's own accepted match is the query.
extern "C" int aps_gplan_filter_mutual(aps_gplan* p) {
  if (!p) APS_FAIL(APS_ERR_ARGS, "", "plan is NULL");
  aps_ctx* c = p->c;
  APS_CTX(c);
  if (p->F == 0) return APS_OK;
  DevBuf<uint8_t> keep;
  APS_TRY(keep.alloc((size_t)p->F, c->stream));
  return aps_k_records_mutual(c->stream, p->records.p, p->img_of_row.p, p->d_off.p, p->F, keep.p);
}

extern "C" int aps_gplan_download_knn(aps_gplan* p, int64_t q0, int64_t q1, uint32_t* idx, float* dist) {
  if (!p || !idx || !dist) APS_FAIL(APS_ERR_ARGS, "", "bad arguments");
  aps_ctx* c = p->c;
  APS_CTX(c);
  if (q0 < 0 || q1 > p->F || q0 > q1) APS_FAIL(APS_ERR_ARGS, "", "query range out of bounds");
  const size_t n = (size_t)(q1 - q0) * p->k;
  if (n) {
    APS_CUDA(cudaMemcpyAsync(idx, p->knn_idx.p + (size_t)q0 * p->k, n * 4, cudaMemcpyDeviceToHost, c->stream));
    APS_CUDA(cudaMemcpyAsync(dist, p->knn_dist.p + (size_t)q0 * p->k, n * 4, cudaMemcpyDeviceToHost, c->stream));
  }
  APS_CUDA(cudaStreamSynchronize(c->stream));
  return APS_OK;
}

extern "C" int aps_gplan_compact(aps_gplan* p) {
  if (!p) APS_FAIL(APS_ERR_ARGS, "", "plan is NULL");
  aps_ctx* c = p->c;
  APS_CTX(c);
  APS_TRY(aps_k_global_compact(c->stream, p->records.p, p->img_of_row.p, p->d_off.p, p->n, p->F, p->dir_counts.p, p->pair_counts.p, p->pair_ptr.p, p->rank.p,
                               p->rows.p));
  p->compacted = true;
  return APS_OK;
}

extern "C" int aps_gplan_pair_counts_device(aps_gplan* p, void** counts_i64) {
  if (!p || !counts_i64 || !p->compacted) APS_FAIL(APS_ERR_ARGS, "", "compact() has not run");
  *counts_i64 = p->pair_counts.p;
  return APS_OK;
}

extern "C" int aps_gplan_download(aps_gplan* p, aps_matchlist** out) {
  if (!p || !out) APS_FAIL(APS_ERR_ARGS, "", "bad arguments");
  aps_ctx* c = p->c;
  APS_CTX(c);
  aps_matchlist* m = new (std::nothrow) aps_matchlist();
  if (!m) APS_FAIL(APS_ERR_ALLOC, "", "out of host memory");
  m->n = p->n;
  const size_t cells = (size_t)p->n * p->n;
  m->pair_ptr.assign(cells + 1, 0);
  if (p->n > 0 && p->compacted) {
    cudaError_t e = cudaMemcpyAsync(m->pair_ptr.data(), p->pair_ptr.p, (cells + 1) * 8, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) {
      delete m;
      APS_FAIL(APS_ERR_CUDA, "", "download failed: %s", cudaGetErrorString(e));
    }
    m->total = m->pair_ptr[cells];
    m->rows.resize((size_t)m->total * 2);
    if (m->total > 0) {
      e = cudaMemcpyAsync(m->rows.data(), p->rows.p, (size_t)m->total * 8, cudaMemcpyDeviceToHost, c->stream);
      if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
      if (e != cudaSuccess) {
        delete m;
        APS_FAIL(APS_ERR_CUDA, "", "download failed: %s", cudaGetErrorString(e));
      }
    }
  } else {
    APS_CUDA(cudaStreamSynchronize(c->stream));
  }
  if (p->dtype == APS_F32 && p->tensor) c->stats[1] = c->h_flags[32];
  if (p->dtype == APS_F32 && p->F > 0) {
    int32_t fl[8];
    if (cudaMemcpy(fl, p->fs.flags.p, sizeof fl, cudaMemcpyDeviceToHost) == cudaSuccess) c->stats[3] = fl[0];
  }
  *out = m;
  return APS_OK;
}

// ------------------------------------------------------------------------------------------------
// featureMatchingGlobal : one call
extern "C" int aps_feature_matching_global(aps_ctx* c, const void* const* desc, const int64_t* counts, int n, int D,
                                           int dtype, int layout, int k, double ratio, int use_bf,
                                           aps_matchlist** out) {
  (void)use_bf;
  return feature_matching_global_impl(c, desc, counts, n, D, dtype, layout, k, ratio, /*mutual*/ 0, out);
}

// the single-context pipeline behind aps_feature_matching_global (and a one-member aps_group); mutual != 0 adds the
// opt-in cross-check of aps_gplan_filter_mutual
int feature_matching_global_impl(aps_ctx* c, const void* const* desc, const int64_t* counts, int n, int D, int dtype,
                                 int layout, int k, double ratio, int mutual, aps_matchlist** out, bool dev) {
  APS_CTX(c);
  if (!out) APS_FAIL(APS_ERR_ARGS, "", "out is NULL");
  *out = nullptr;
  aps_gplan* p = nullptr;
  APS_TRY(aps_gplan_create(c, counts, n, D, dtype, k, &p));
  int rc = APS_OK;
  if (p->F > 0) rc = gplan_run(p, desc, layout, ratio, mutual, dev);  // featureMatchingGlobal.m:49-52,65-67: all empty -> cell(numImg)
  if (rc == APS_OK) rc = aps_gplan_download(p, out);
  aps_gplan_destroy(p);
  return rc;
}

int gplan_run(aps_gplan* p, const void* const* desc, int layout, double ratio, int mutual, bool dev) {
  if (dev)  // the pooled device matrix of the set: one copy into the plan
    APS_CUDA(cudaMemcpyAsync(aps_gplan_desc_device(p), desc[0], (size_t)p->F * p->D * (p->dtype == APS_F32 ? 4 : 1),
                             cudaMemcpyDeviceToDevice, p->c->stream));
  else
    APS_TRY(aps_gplan_upload(p, desc, layout));
  APS_TRY(aps_gplan_prepare(p));
  APS_TRY(aps_gplan_knn(p, 0, p->F));
  APS_TRY(aps_gplan_filter(p, 0, p->F, ratio));
  if (mutual) APS_TRY(aps_gplan_filter_mutual(p));
  return aps_gplan_compact(p);
}

void gplan_lists(aps_gplan* p, GlobalLists& L) {
  L.plan = p;
  L.order.assign(1, 0);
  L.cell_off = {0, (int64_t)p->n * p->n};
  L.pair_counts = p->pair_counts.p;
  L.pair_ptr = p->pair_ptr.p;
  L.rows = p->rows.p;
  L.F = p->F;
  L.Ft = p->dtype == APS_F32 && p->tensor ? p->F : 0;
}

// Same with the pooled descriptors ALREADY ON THE DEVICE (a GPU extractor's output, or a previous stage's buffer): the
// one-set case of aps_feature_matching_global_sets_dev, the context checked first as it always was.
extern "C" int aps_feature_matching_global_dev(aps_ctx* c, const void* d_pooled, const int64_t* counts, int n, int D,
                                               int dtype, int k, double ratio, int mutual, aps_matchlist** out) {
  APS_CTX(c);
  if (!out) APS_FAIL(APS_ERR_ARGS, "", "out is NULL");
  return aps_feature_matching_global_sets_dev(c, 1, &n, d_pooled, counts, D, dtype, k, ratio, 0, mutual, nullptr, out);
}

// ------------------------------------------------------------------------------------------------
// imageMatching.m:75-100: the one-set case of aps_select_partners_sets (pairs_lin may be NULL here)
extern "C" int aps_select_partners(aps_ctx* c, const int64_t* counts, int n, int m, uint8_t* cand,
                                   int64_t* pairs_lin, int64_t* npairs) {
  APS_CTX(c);
  if (n < 0 || (n > 0 && (!counts || !cand))) APS_FAIL(APS_ERR_ARGS, "", "bad arguments");
  std::vector<int64_t> scratch(pairs_lin ? 0 : (size_t)n * (n - 1) / 2 + 1);
  int64_t set_pair_ptr[2] = {0, 0};
  APS_TRY(aps_select_partners_sets(c, 1, &n, counts, m, cand, pairs_lin ? pairs_lin : scratch.data(), set_pair_ptr));
  if (npairs) *npairs = set_pair_ptr[1];
  return APS_OK;
}

// imageMatching.m:75-100 for nsets sets: one upload (counts and the set tables), K6 over every set's block, the
// device-side find(), one download, whatever nsets
extern "C" int aps_select_partners_sets(aps_ctx* c, int nsets, const int* set_images, const int64_t* counts, int m,
                                        uint8_t* cand, int64_t* pairs_lin, int64_t* set_pair_ptr) {
  std::vector<int64_t> img0;
  APS_TRY(sets_image_offsets(nsets, set_images, img0));
  if (!set_pair_ptr) APS_FAIL(APS_ERR_ARGS, "", "set_pair_ptr is NULL");
  int64_t cells = 0, pair_cap = 0;
  for (int b = 0; b < nsets; ++b) {
    const int64_t n = set_images[b];
    cells += n * n;
    pair_cap += n * (n - 1) / 2;
  }
  if (cells > 0 && (!counts || !cand || !pairs_lin)) APS_FAIL(APS_ERR_ARGS, "", "NULL argument");
  APS_CTX(c);
  for (int b = 0; b <= nsets; ++b) set_pair_ptr[b] = 0;
  if (cells == 0) return APS_OK;
  // host / device layout [set_img | cell_off (nsets + 1 each) | counts (cells)], results [set_pair_ptr | pairs_lin | cand]
  const size_t nt = (size_t)nsets + 1, in_words = 2 * nt + (size_t)cells, out_words = nt + (size_t)pair_cap;
  std::vector<int64_t> in(in_words);
  std::copy(img0.begin(), img0.end(), in.begin());
  in[nt] = 0;
  for (int b = 0; b < nsets; ++b) in[nt + b + 1] = in[nt + b] + (int64_t)set_images[b] * set_images[b];
  std::memcpy(in.data() + 2 * nt, counts, (size_t)cells * 8);
  cudaStream_t s = c->stream;
  DevBuf<int64_t> din, dout;
  APS_TRY(din.alloc(in_words, s));
  APS_TRY(dout.alloc(out_words + aps_ceil_div(cells, 8), s));
  uint8_t* dcand = (uint8_t*)(dout.p + out_words);
  uint8_t* h = (uint8_t*)aps_ctx_stage(c, out_words * 8 + (size_t)cells);
  if (!h) APS_FAIL(APS_ERR_ALLOC, "", "pinned staging allocation failed");
  APS_CUDA(cudaMemcpyAsync(din.p, in.data(), in_words * 8, cudaMemcpyHostToDevice, s));
  APS_TRY(aps_k_select_partners_sets(s, din.p + 2 * nt, (int)img0[nsets], cells, din.p, din.p + nt, nsets, m, dcand));
  APS_TRY(aps_k_select_compact(s, dcand, cells, din.p + nt, nsets, dout.p + nt, dout.p));
  APS_CUDA(cudaMemcpyAsync(h, dout.p, out_words * 8 + (size_t)cells, cudaMemcpyDeviceToHost, s));
  APS_CUDA(cudaStreamSynchronize(s));  // `in` stays alive until here
  const int64_t* hw = (const int64_t*)h;
  std::memcpy(set_pair_ptr, hw, nt * 8);
  std::memcpy(pairs_lin, hw + nt, (size_t)hw[nsets] * 8);
  std::memcpy(cand, h + out_words * 8, (size_t)cells);
  return APS_OK;
}

// ------------------------------------------------------------------------------------------------
// diagnostics: run the tcgen05 candidate kernel alone and return what its epilogue saw
extern "C" int aps_debug_tc_slots(aps_ctx* c, int64_t nq, int64_t nt) {
  return c ? aps_k_knn_tc_slots(c->sm_count, nq, 0, nt) : 0;
}
extern "C" int aps_debug_tc_scores(aps_ctx* c, const float* Q, int64_t nq, const float* T, int64_t nt, int D,
                                   int nseg, float* scores, uint32_t* cand_idx, float* cand_score) {
  APS_CTX(c);
  (void)nseg;
  if (!Q || !T || nq <= 0 || nt <= 0 || D <= 0) APS_FAIL(APS_ERR_ARGS, "", "bad arguments");
  const int nslot = aps_k_knn_tc_slots(c->sm_count, nq, 0, nt);
  const int Dp = (D + 63) / 64 * 64;
  if (!aps_k_knn_tc_supported(Dp)) APS_FAIL(APS_ERR_DIM, "", "unsupported descriptor length %d", D);
  FloatSet qs, ts;
  DevBuf<uint8_t> tmp;
  APS_TRY(floatset_alloc(c, qs, nq, D));
  APS_TRY(floatset_alloc(c, ts, nt, D));
  APS_TRY(floatset_reset_flags(c, ts));
  APS_TRY(stage_matrix(c, Q, nq, D, 4, APS_ROW_MAJOR, qs.raw.p, tmp));
  APS_TRY(stage_matrix(c, T, nt, D, 4, APS_ROW_MAJOR, ts.raw.p, tmp));
  APS_TRY(aps_k_prepare_norm(c->stream, qs.raw.p, nq, D, APS_NORM_NONE, qs.raw.p, qs.sq.p, qs.invn.p, ts.flags.p));
  APS_TRY(aps_k_prepare_norm(c->stream, ts.raw.p, nt, D, APS_NORM_NONE, ts.raw.p, ts.sq.p, ts.invn.p, ts.flags.p));
  APS_TRY(qs.xb.alloc((size_t)nq * Dp, c->stream));
  APS_TRY(qs.colscale.alloc((size_t)nq + 256, c->stream));
    APS_TRY(qs.colbias.alloc((size_t)nq + 256, c->stream));
  APS_TRY(ts.xb.alloc((size_t)nt * Dp, c->stream));
  APS_TRY(ts.colscale.alloc((size_t)nt + 256, c->stream));
    APS_TRY(ts.colbias.alloc((size_t)nt + 256, c->stream));
  APS_TRY(aps_k_prepare_operands(c->stream, qs.raw.p, qs.raw.p, qs.sq.p, qs.invn.p, nq, D, Dp, ts.flags.p, 1, qs.xb.p, qs.colscale.p, qs.colbias.p));
  APS_TRY(aps_k_prepare_operands(c->stream, ts.raw.p, ts.raw.p, ts.sq.p, ts.invn.p, nt, D, Dp, ts.flags.p, 1, ts.xb.p, ts.colscale.p, ts.colbias.p));
  DevBuf<float> dump, cscore;
  DevBuf<uint32_t> cidx;
  if (scores) APS_TRY(dump.alloc((size_t)nq * nt, c->stream));
  APS_TRY(cidx.alloc((size_t)nq * nslot * 8, c->stream));
  APS_TRY(cscore.alloc((size_t)nq * nslot * 8, c->stream));
  aps_tc_problem p;
  APS_TRY(floatset_finish_train(c, ts, /*sort*/ false));  // natural column order: the dump is indexed by column
  p.Qb = qs.xb.p; p.Tb = ts.xb.p; p.colscale = ts.colscale.p; p.colbias = ts.colbias.p; p.tile_bounds = ts.tile_bounds.p;
  p.bias = 1;
  p.Fq_total = nq; p.Ft_total = nt; p.Dp = Dp;
  p.q0 = 0; p.q1 = nq; p.t0 = 0; p.t1 = nt;
  p.nslot = nslot; p.kcand = 8;
  p.cand_idx = cidx.p; p.cand_score = cscore.p;
  p.dump = scores ? dump.p : nullptr;
  APS_TRY(aps_k_knn_tc(c->stream, c->sm_count, p));
  if (scores) APS_CUDA(cudaMemcpyAsync(scores, dump.p, (size_t)nq * nt * 4, cudaMemcpyDeviceToHost, c->stream));
  if (cand_idx) APS_CUDA(cudaMemcpyAsync(cand_idx, cidx.p, (size_t)nq * nslot * 8 * 4, cudaMemcpyDeviceToHost, c->stream));
  if (cand_score) APS_CUDA(cudaMemcpyAsync(cand_score, cscore.p, (size_t)nq * nslot * 8 * 4, cudaMemcpyDeviceToHost, c->stream));
  APS_CUDA(cudaStreamSynchronize(c->stream));
  return APS_OK;
}

// diagnostics: the candidate lists of one tcgen05 launch, with the operands, constants and schedule it ran on.  The
// preparation and the launch are the ones of float_knn for a search of k neighbours: prep 0 = the global plan
// (APS_NORM_GLOBAL, fp16 operands, scale-only scores), prep 1 = flann_knn_win (raw rows, bf16, bias -|t|^2/2);
// rows != NULL = its second pass.
extern "C" int aps_debug_tc_candidates_k(aps_ctx* c, const float* Q, int64_t nq, const float* T, int64_t nt, int D,
                                         int prep, int natural_order, int64_t q0, int64_t q1, int64_t t0, int64_t t1,
                                         const int32_t* rows, int64_t nrows, uint32_t* cand_idx, float* cand_score,
                                         int32_t* perm, uint16_t* q_bits, uint16_t* t_bits, float* colscale,
                                         float* colbias, int64_t* info, int k) {
  APS_CTX(c);
  if (!Q || !T || nq <= 0 || nt <= 0 || D <= 0 || (prep != 0 && prep != 1) || !cand_idx || !cand_score || !perm ||
      !q_bits || !t_bits || !colscale || !colbias || !info)
    APS_FAIL(APS_ERR_ARGS, "", "bad arguments");
  if (k < 1 || k > kTcMaxK) APS_FAIL(APS_ERR_K, "", "the tensor path serves 1 <= k <= %d (got %d)", kTcMaxK, k);
  if (q0 < 0 || q1 > nq || q0 >= q1 || t0 < 0 || t1 > nt || t0 >= t1) APS_FAIL(APS_ERR_ARGS, "", "range out of bounds");
  if (rows && (nrows < 0 || nrows > q1 - q0)) APS_FAIL(APS_ERR_ARGS, "", "more listed rows than the query range holds");
  const int Dp = (D + 63) / 64 * 64;
  if (!aps_k_knn_tc_supported(Dp)) APS_FAIL(APS_ERR_DIM, "", "unsupported descriptor length %d", D);
  if (rows)
    for (int64_t i = 0; i < nrows; ++i)
      if (rows[i] < q0 || rows[i] >= q1) APS_FAIL(APS_ERR_ARGS, "", "listed row %lld outside the query range", (long long)rows[i]);
  cudaStream_t s = c->stream;
  const bool self = (Q == T && nq == nt), global = prep == 0;
  const int norm_mode = global ? APS_NORM_GLOBAL : APS_NORM_NONE, bias_mode = global ? 0 : 1;
  FloatSet ts, qs;
  DevBuf<uint8_t> tmp;
  ts.fp16 = qs.fp16 = global;  // as aps_gplan_create
  APS_TRY(floatset_alloc(c, ts, nt, D));
  APS_TRY(floatset_reset_flags(c, ts));
  APS_TRY(stage_matrix(c, T, nt, D, 4, APS_ROW_MAJOR, ts.raw.p, tmp));
  if (!self) {
    APS_TRY(floatset_alloc(c, qs, nq, D));
    APS_TRY(stage_matrix(c, Q, nq, D, 4, APS_ROW_MAJOR, qs.raw.p, tmp));
  }
  // both flag passes (shared flag words) before the operands of either side, as flann_knn_win
  FloatSet* sides[2] = {&ts, self ? nullptr : &qs};
  for (FloatSet* f : sides) {
    if (!f) continue;
    if (norm_mode != APS_NORM_NONE) APS_TRY(f->xn.alloc((size_t)f->N * D, s));
    APS_TRY(aps_k_prepare_norm(s, f->raw.p, f->N, D, norm_mode, f->xn.p ? f->xn.p : f->raw.p, f->sq.p, f->invn.p,
                               ts.flags.p, f->fp16));
  }
  for (FloatSet* f : sides) {
    if (!f) continue;
    APS_TRY(f->xb.alloc((size_t)f->N * Dp, s));
    APS_TRY(f->colscale.alloc((size_t)f->N + 256, s));
    APS_TRY(f->colbias.alloc((size_t)f->N + 256, s));
    APS_TRY(aps_k_prepare_operands(s, f->raw.p, f->xn.p ? f->xn.p : f->raw.p, f->sq.p, f->invn.p, f->N, D, Dp, ts.flags.p,
                                   bias_mode, f->xb.p, f->colscale.p, f->colbias.p, f->fp16));
  }
  APS_TRY(floatset_finish_train(c, ts, !natural_order));
  const FloatSide qv = self ? ts.side() : qs.side(), tv = ts.side();
  aps_tc_problem p;
  p.Qb = qv.xb; p.Tb = tv.xb_t; p.colscale = tv.colscale_t; p.colbias = tv.colbias_t; p.tile_bounds = tv.tile_bounds;
  p.bias = bias_mode;
  p.Fq_total = nq; p.Ft_total = nt; p.Dp = Dp;
  p.q0 = q0; p.q1 = q1; p.t0 = t0; p.t1 = t1;
  p.kcand = tc_list_length(k);
  p.dump = nullptr;
  p.operand_fp16 = global ? 2 : 0;
  p.exact_flag = ts.flags.p;
  const int64_t nr = q1 - q0;
  DevBuf<int32_t> drows;
  DevBuf<__nv_bfloat16> qb2;
  if (rows) {  // float_knn's second pass: the listed rows gathered into a compact query matrix, count on the device
    const int32_t cnt = (int32_t)nrows;
    APS_TRY(drows.alloc((size_t)nr + 1, s));
    APS_TRY(qb2.alloc((size_t)nr * Dp, s));
    if (nrows > 0) APS_CUDA(cudaMemcpyAsync(drows.p, rows, (size_t)nrows * 4, cudaMemcpyHostToDevice, s));
    APS_CUDA(cudaMemcpyAsync(drows.p + nr, &cnt, 4, cudaMemcpyHostToDevice, s));
    APS_TRY(aps_k_gather_rows(s, qv.xb, Dp, drows.p, drows.p + nr, nr, qb2.p));
    p.Qb = qb2.p; p.Fq_total = nr; p.q0 = 0; p.q1 = nr;
    p.nrows_dev = drows.p + nr;
  }
  p.nslot = aps_k_knn_tc_slots(c->sm_count, nr, t0, t1, rows ? 1 : 0);
  int d[7];
  APS_TRY(aps_k_knn_tc_describe(c->sm_count, p, d));
  DevBuf<uint32_t> cidx;
  DevBuf<float> cscore;
  const size_t ncand = (size_t)nr * p.nslot * p.kcand;
  APS_TRY(cidx.alloc(ncand, s));
  APS_TRY(cscore.alloc(ncand, s));
  APS_CUDA(cudaMemsetAsync(cidx.p, 0xA5, ncand * 4, s));    // 0xA5A5A5A5: never a train position of these sizes
  APS_CUDA(cudaMemsetAsync(cscore.p, 0xFF, ncand * 4, s));  // NaN
  p.cand_idx = cidx.p; p.cand_score = cscore.p;
  APS_TRY(aps_k_knn_tc(s, c->sm_count, p));
  int32_t exact = 0;
  APS_CUDA(cudaMemcpyAsync(&exact, ts.flags.p, 4, cudaMemcpyDeviceToHost, s));
  APS_CUDA(cudaMemcpyAsync(cand_idx, cidx.p, ncand * 4, cudaMemcpyDeviceToHost, s));
  APS_CUDA(cudaMemcpyAsync(cand_score, cscore.p, ncand * 4, cudaMemcpyDeviceToHost, s));
  if (tv.perm) APS_CUDA(cudaMemcpyAsync(perm, tv.perm, (size_t)nt * 4, cudaMemcpyDeviceToHost, s));
  APS_CUDA(cudaMemcpy2DAsync(q_bits, (size_t)D * 2, qv.xb, (size_t)Dp * 2, (size_t)D * 2, (size_t)nq, cudaMemcpyDeviceToHost, s));
  APS_CUDA(cudaMemcpy2DAsync(t_bits, (size_t)D * 2, ts.xb.p, (size_t)Dp * 2, (size_t)D * 2, (size_t)nt, cudaMemcpyDeviceToHost, s));
  APS_CUDA(cudaMemcpyAsync(colscale, ts.colscale.p, (size_t)nt * 4, cudaMemcpyDeviceToHost, s));
  APS_CUDA(cudaMemcpyAsync(colbias, ts.colbias.p, (size_t)nt * 4, cudaMemcpyDeviceToHost, s));
  APS_CUDA(cudaStreamSynchronize(s));
  if (!tv.perm)
    for (int64_t i = 0; i < nt; ++i) perm[i] = (int32_t)i;
  // float_knn: rows of full-width units are re-ranked from list 0 alone (first pass only)
  const int64_t rows_full = (!rows && p.nslot > 1) ? aps_k_knn_tc_full_rows(c->sm_count, nr, t0, t1) : 0;
  const int64_t v[12] = {c->sm_count, d[0], rows_full, exact, p.operand_fp16, d[1], d[2], d[3], d[4], d[5], d[6],
                         p.kcand};
  memcpy(info, v, sizeof v);
  return APS_OK;
}

extern "C" int aps_debug_tc_candidates(aps_ctx* c, const float* Q, int64_t nq, const float* T, int64_t nt, int D,
                                       int prep, int natural_order, int64_t q0, int64_t q1, int64_t t0, int64_t t1,
                                       const int32_t* rows, int64_t nrows, uint32_t* cand_idx, float* cand_score,
                                       int32_t* perm, uint16_t* q_bits, uint16_t* t_bits, float* colscale,
                                       float* colbias, int64_t* info) {
  int64_t v[12];
  APS_TRY(aps_debug_tc_candidates_k(c, Q, nq, T, nt, D, prep, natural_order, q0, q1, t0, t1, rows, nrows, cand_idx,
                                    cand_score, perm, q_bits, t_bits, colscale, colbias, info ? v : nullptr, 4));
  memcpy(info, v, 11 * sizeof(int64_t));
  return APS_OK;
}

// diagnostics: the fp16 screen of ONE (query set, train set) pair, with the raw accumulator registers
extern "C" int aps_debug_pair_screen(aps_ctx* c, const float* A, int64_t N1, const float* B, int64_t N2, int D,
                                     float* b1b2, uint32_t* dump, int dump_tiles) {
  APS_CTX(c);
  if (!A || !B || N1 <= 0 || N2 <= 0 || D <= 0 || !b1b2) APS_FAIL(APS_ERR_ARGS, "", "bad arguments");
  const int Dp = (D + 63) / 64 * 64;
  if (!aps_k_knn_tc_supported(Dp)) APS_FAIL(APS_ERR_DIM, "", "unsupported descriptor length %d", D);
  cudaStream_t s = c->stream;
  const int64_t F = N1 + N2;
  DevBuf<float> raw;
  DevBuf<uint16_t> xh;
  DevBuf<uint32_t> scr, ddump;
  DevBuf<aps_tc_unit> units;
  DevBuf<int32_t> tab;
  DevBuf<int64_t> off2;
  APS_TRY(raw.alloc((size_t)F * D, s));
  APS_TRY(xh.alloc((size_t)F * Dp, s));
  APS_TRY(scr.alloc((size_t)N1, s));
  const int64_t U = (N1 + 255) / 256;
  APS_TRY(units.alloc((size_t)U, s));
  if (dump && dump_tiles > 0) {
    APS_TRY(ddump.alloc((size_t)N1 * dump_tiles * 64, s));
    APS_CUDA(cudaMemsetAsync(ddump.p, 0, (size_t)N1 * dump_tiles * 64 * 4, s));
  }
  APS_CUDA(cudaMemcpyAsync(raw.p, A, (size_t)N1 * D * 4, cudaMemcpyHostToDevice, s));
  APS_CUDA(cudaMemcpyAsync(raw.p + (size_t)N1 * D, B, (size_t)N2 * D * 4, cudaMemcpyHostToDevice, s));
  APS_TRY(aps_k_prepare_operands_f16(s, raw.p, F, D, Dp, xh.p));
  const int32_t htab[5] = {0, (int32_t)N1, (int32_t)N1, (int32_t)N2, 1};
  const int64_t hoff[4] = {0, N1, 0, U};
  APS_TRY(tab.alloc(5, s));
  APS_TRY(off2.alloc(4, s));
  APS_CUDA(cudaMemcpyAsync(tab.p, htab, sizeof htab, cudaMemcpyHostToDevice, s));
  APS_CUDA(cudaMemcpyAsync(off2.p, hoff, sizeof hoff, cudaMemcpyHostToDevice, s));
  aps_pair_screen_tables t;
  t.qoff = tab.p; t.qcnt = tab.p + 1; t.toff = tab.p + 2; t.tcnt = tab.p + 3; t.timg = tab.p + 4;
  t.eoff = off2.p; t.uoff = off2.p + 2; t.npairs = 1;
  APS_TRY(aps_k_pair_screen(s, c->sm_count, xh.p, F, xh.p, F, Dp, t, units.p, U, scr.p, ddump.p, ddump.p ? dump_tiles : 0));
  std::vector<uint32_t> h((size_t)N1);
  APS_CUDA(cudaMemcpyAsync(h.data(), scr.p, (size_t)N1 * 4, cudaMemcpyDeviceToHost, s));
  if (ddump.p) APS_CUDA(cudaMemcpyAsync(dump, ddump.p, (size_t)N1 * dump_tiles * 64 * 4, cudaMemcpyDeviceToHost, s));
  APS_CUDA(cudaStreamSynchronize(s));
  for (int64_t i = 0; i < N1; ++i) {   // unpack the two fp16 values (pure bit manipulation, no arithmetic)
    for (int w = 0; w < 2; ++w) {
      const uint16_t hb = (uint16_t)(h[(size_t)i] >> (16 * w));
      const uint32_t sign = (uint32_t)(hb & 0x8000u) << 16, ex = (hb >> 10) & 0x1fu, man = hb & 0x3ffu;
      uint32_t f;
      if (ex == 0) {
        if (man == 0) f = sign;
        else {
          int e = -1;
          uint32_t m = man;
          do { ++e; m <<= 1; } while (!(m & 0x400u));
          f = sign | ((uint32_t)(127 - 15 - e) << 23) | ((m & 0x3ffu) << 13);
        }
      } else if (ex == 31) f = sign | 0x7f800000u | (man << 13);
      else f = sign | ((ex + 112u) << 23) | (man << 13);
      memcpy(&b1b2[2 * i + w], &f, 4);
    }
  }
  return APS_OK;
}
