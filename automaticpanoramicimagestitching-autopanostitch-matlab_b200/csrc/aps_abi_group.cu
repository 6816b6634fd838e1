// aps_abi_group.cu -- single-process multi-GPU matching: a device group (one aps_ctx per listed GPU) and the one-call
// global / pairwise entries that run the staged plans of aps_abi.cu / aps_abi_pairwise.cu on every member at once.
// One host thread per member issues all of that member's calls (the pairwise batches synchronise on pageable host
// tables, so a single issuing thread would serialise the GPUs).  The exchanges between members are device-to-device
// copies (cudaMemcpyPeerAsync; the driver stages them where peer access is not available), ordered with events.
// A one-member group runs the single-context pipelines unchanged.
#include <algorithm>
#include <functional>
#include <new>
#include <string>
#include <thread>

#include "aps_abi_internal.cuh"

namespace {

// per-member stage timestamps of the last group call (aps_group_stage_times)
enum { EV_START, EV_UPLOAD, EV_EXCHANGE, EV_SEARCH, EV_GATHER, EV_FINISH, EV_COUNT };

struct MemberStatus {
  int rc = APS_OK;
  std::string msg, id;
};

}  // namespace

struct aps_group {
  std::vector<aps_ctx*> ctx;
  std::vector<std::vector<cudaEvent_t>> ev;  // [member][EV_*]
  std::vector<int> recorded;                 // highest EV_* recorded + 1 by the last call, per member
};

// Runs fn(i) for every member on its own host thread, joins them all, and carries the first failing member's status,
// message and MATLAB id over to the calling thread (aps_last_error / aps_error_id are thread-local).
static int run_members(aps_group* g, const std::function<int(int)>& fn) {
  const int N = (int)g->ctx.size();
  std::vector<MemberStatus> st((size_t)N);
  auto body = [&](int i) {
    st[i].rc = fn(i);
    if (st[i].rc != APS_OK) {
      st[i].msg = aps_last_error();
      st[i].id = aps_error_id();
    }
  };
  if (N == 1) {
    body(0);
  } else {
    std::vector<std::thread> th;
    th.reserve((size_t)N);
    for (int i = 0; i < N; ++i) th.emplace_back(body, i);
    for (std::thread& t : th) t.join();
  }
  for (int i = 0; i < N; ++i)
    if (st[i].rc != APS_OK) {
      aps_set_error(st[i].rc, st[i].id.c_str(), "device group member %d (GPU %d): %s", i, g->ctx[i]->device,
                    st[i].msg.c_str());
      return st[i].rc;
    }
  return APS_OK;
}

static int record(aps_group* g, int i, int which) {
  APS_CUDA(cudaEventRecord(g->ev[i][which], g->ctx[i]->stream));
  g->recorded[i] = std::max(g->recorded[i], which + 1);
  return APS_OK;
}

// Every member's stream drains before any plan is released: a member's buffers may still be the source of another
// member's copy.
static void drain(aps_group* g) {
  run_members(g, [&](int i) -> int {
    cudaSetDevice(g->ctx[i]->device);
    cudaStreamSynchronize(g->ctx[i]->stream);
    return APS_OK;
  });
}

// Lets member i read and write member j's memory directly wherever cudaDeviceCanAccessPeer allows.  Everything a group
// exchanges (descriptor matrices, records) is a plan buffer from the device's default stream-ordered pool
// (DevBuf: cudaMallocAsync), and pool memory is reachable from a peer only once the owning pool grants access
// (cudaMemPoolSetAccess); cudaDeviceEnablePeerAccess covers cudaMalloc'd memory.  Both are granted.
static int enable_peer_access(const int* devices, int ndev) {
  for (int i = 0; i < ndev; ++i)
    for (int j = 0; j < ndev; ++j) {
      int can = 0;
      if (devices[i] == devices[j]) continue;
      APS_CUDA(cudaDeviceCanAccessPeer(&can, devices[i], devices[j]));
      if (!can) continue;
      APS_CUDA(cudaSetDevice(devices[i]));
      const cudaError_t e = cudaDeviceEnablePeerAccess(devices[j], 0);
      if (e == cudaErrorPeerAccessAlreadyEnabled)
        (void)cudaGetLastError();
      else
        APS_CUDA(e);
      cudaMemPool_t pool;  // device j's pool: accessible from device i
      APS_CUDA(cudaDeviceGetDefaultMemPool(&pool, devices[j]));
      cudaMemAccessDesc acc = {};
      acc.location.type = cudaMemLocationTypeDevice;
      acc.location.id = devices[i];
      acc.flags = cudaMemAccessFlagsProtReadWrite;
      APS_CUDA(cudaMemPoolSetAccess(pool, &acc, 1));
    }
  return APS_OK;
}

static int group_create(const int* devices, int ndev, bool shared, aps_group** out) {
  if (!out) APS_FAIL(APS_ERR_ARGS, "", "aps_group_create: out is NULL");
  *out = nullptr;
  if (!devices || ndev < 1) APS_FAIL(APS_ERR_ARGS, "", "aps_group_create: the device list is empty");
  for (int i = 0; i < ndev; ++i) {
    if (devices[i] < 0) APS_FAIL(APS_ERR_ARGS, "", "device %d is negative", devices[i]);
    for (int j = 0; j < i && !shared; ++j)
      if (devices[j] == devices[i]) APS_FAIL(APS_ERR_ARGS, "", "device %d is listed twice", devices[i]);
  }
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0)
    APS_FAIL(APS_ERR_NOGPU, "apsmatch:nogpu", "no CUDA device available (%s); libapsmatch has no CPU fallback",
             e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
  for (int i = 0; i < ndev; ++i)
    if (devices[i] >= count) APS_FAIL(APS_ERR_ARGS, "", "device %d out of range (0..%d)", devices[i], count - 1);
  aps_group* g = new (std::nothrow) aps_group();
  if (!g) APS_FAIL(APS_ERR_ALLOC, "", "out of host memory");
  for (int i = 0; i < ndev; ++i) {
    aps_ctx* c = nullptr;
    int rc = aps_ctx_create(devices[i], &c);
    if (rc == APS_OK) {
      g->ctx.push_back(c);
      g->ev.emplace_back(EV_COUNT, nullptr);
      g->recorded.push_back(0);
      for (int k = 0; k < EV_COUNT && rc == APS_OK; ++k)
        if (cudaEventCreate(&g->ev.back()[k]) != cudaSuccess) {
          aps_set_error(APS_ERR_CUDA, "", "cudaEventCreate failed on device %d", devices[i]);
          rc = APS_ERR_CUDA;
        }
    }
    if (rc != APS_OK) {
      const std::string msg = aps_last_error(), id = aps_error_id();
      aps_group_destroy(g);
      aps_set_error(rc, id.c_str(), "%s", msg.c_str());
      return rc;
    }
  }
  // Direct peer access where the topology allows it; elsewhere the driver stages the copies through the host.
  const int rc = enable_peer_access(devices, ndev);
  if (rc != APS_OK) {
    const std::string msg = aps_last_error();
    aps_group_destroy(g);
    aps_set_error(rc, "", "%s", msg.c_str());
    return rc;
  }
  *out = g;
  return APS_OK;
}

extern "C" int aps_group_create(const int* devices, int ndev, aps_group** out) {
  return group_create(devices, ndev, false, out);
}

// Test hook: nmembers contexts on ONE device run the multi-member pipeline (threads, events, device-to-device copies,
// merge) where only one GPU is available.
extern "C" int aps_debug_group_create_shared(int device, int nmembers, aps_group** out) {
  if (nmembers < 1 || nmembers > 64) APS_FAIL(APS_ERR_ARGS, "", "nmembers must be 1..64");
  std::vector<int> devs((size_t)nmembers, device);
  return group_create(devs.data(), nmembers, true, out);
}

extern "C" void aps_group_destroy(aps_group* g) {
  if (!g) return;
  for (size_t i = 0; i < g->ctx.size(); ++i) {
    cudaSetDevice(g->ctx[i]->device);
    for (cudaEvent_t e : g->ev[i])
      if (e) cudaEventDestroy(e);
    aps_ctx_destroy(g->ctx[i]);
  }
  delete g;
}

extern "C" int aps_group_size(const aps_group* g) { return g ? (int)g->ctx.size() : 0; }

extern "C" aps_ctx* aps_group_ctx(aps_group* g, int i) {
  if (!g || i < 0 || i >= (int)g->ctx.size()) return nullptr;
  return g->ctx[i];
}

extern "C" int aps_group_stage_times(aps_group* g, int i, double ms[4]) {
  if (!g || !ms || i < 0 || i >= (int)g->ctx.size()) APS_FAIL(APS_ERR_ARGS, "", "bad arguments");
  APS_CUDA(cudaSetDevice(g->ctx[i]->device));
  APS_CUDA(cudaStreamSynchronize(g->ctx[i]->stream));
  // upload, exchange, search, finish = consecutive intervals between the recorded events
  for (int s = 0; s < 4; ++s) {
    ms[s] = 0.0;
    const int a = s, b = s == 3 ? EV_FINISH : s + 1;
    if (g->recorded[i] <= b) continue;
    float t = 0.f;
    APS_CUDA(cudaEventElapsedTime(&t, g->ev[i][a], g->ev[i][b]));
    ms[s] = t;
  }
  return APS_OK;
}

// ------------------------------------------------------------------------------------------------
// featureMatchingGlobal across the members: every member holds all descriptors, searches its block of query rows and
// files its records; member 0 gathers the record slices and compacts.
extern "C" int aps_group_feature_matching_global(aps_group* g, const void* const* desc, const int64_t* counts, int n,
                                                 int D, int dtype, int layout, int k, double ratio, int mutual,
                                                 aps_matchlist** out) {
  if (!g || g->ctx.empty()) APS_FAIL(APS_ERR_NOGPU, "apsmatch:nogpu", "device group is NULL (no GPU context; there is no CPU path)");
  if (!out) APS_FAIL(APS_ERR_ARGS, "", "out is NULL");
  *out = nullptr;
  const int N = (int)g->ctx.size();
  std::fill(g->recorded.begin(), g->recorded.end(), 0);
  if (N == 1) return feature_matching_global_impl(g->ctx[0], desc, counts, n, D, dtype, layout, k, ratio, mutual, out);
  if (n < 0 || (n > 0 && !counts)) APS_FAIL(APS_ERR_ARGS, "", "bad arguments");

  // image ranges of the uploads (contiguous, balanced by row count) and the query-row blocks of the search
  // (multigpu.shard_bounds: equal multiples of 128 rows, members past F get an empty block)
  std::vector<int64_t> off((size_t)n + 1, 0);
  for (int i = 0; i < n; ++i) off[i + 1] = off[i] + std::max<int64_t>(counts[i], 0);
  const int64_t F = off[n];
  std::vector<int> img0((size_t)N + 1, n);
  img0[0] = 0;
  for (int m = 1, i = 0; m < N; ++m) {
    // image i goes to member floor(N * (row midpoint of i) / F)
    while (i < n && (off[i] + off[i + 1]) * (int64_t)N < 2 * (int64_t)m * F) ++i;
    img0[m] = i;
  }
  const int64_t S = (F + 127) / 128;
  const int64_t rows_per = (S + N - 1) / N * 128;
  auto q_lo = [&](int m) { return std::min(F, (int64_t)m * rows_per); };
  auto q_hi = [&](int m) { return std::min(F, (int64_t)(m + 1) * rows_per); };

  std::vector<aps_gplan*> plan((size_t)N, nullptr);
  const int esz = dtype == APS_F32 ? 4 : 1;
  // 1: plans, each member's share of the host upload
  int rc = run_members(g, [&](int i) -> int {
    APS_TRY(aps_gplan_create(g->ctx[i], counts, n, D, dtype, k, &plan[i]));
    if (F == 0) return APS_OK;
    APS_TRY(record(g, i, EV_START));
    APS_TRY(gplan_upload_images(plan[i], desc, layout, img0[i], img0[i + 1]));
    return record(g, i, EV_UPLOAD);
  });
  // 2: every other member's rows peer-to-peer, then K1 (replicated) and this member's block of the search
  if (rc == APS_OK && F > 0)
    rc = run_members(g, [&](int i) -> int {
      aps_ctx* c = g->ctx[i];
      APS_CTX(c);
      for (int j = 0; j < N; ++j) {
        const int64_t r0 = off[img0[j]], r1 = off[img0[j + 1]];
        if (j == i || r1 == r0) continue;
        APS_CUDA(cudaStreamWaitEvent(c->stream, g->ev[j][EV_UPLOAD], 0));
        const size_t o = (size_t)r0 * D * esz;
        APS_CUDA(cudaMemcpyPeerAsync((char*)aps_gplan_desc_device(plan[i]) + o, c->device,
                                     (const char*)aps_gplan_desc_device(plan[j]) + o, g->ctx[j]->device,
                                     (size_t)(r1 - r0) * D * esz, c->stream));
      }
      APS_TRY(record(g, i, EV_EXCHANGE));
      APS_TRY(aps_gplan_prepare(plan[i]));
      APS_TRY(aps_gplan_knn(plan[i], q_lo(i), q_hi(i)));
      APS_TRY(aps_gplan_filter(plan[i], q_lo(i), q_hi(i), ratio));
      return record(g, i, EV_SEARCH);
    });
  // 3: member 0 gathers the record slices (8 bytes per query row), cross-checks, compacts and downloads
  if (rc == APS_OK)
    rc = run_members(g, [&](int i) -> int {
      if (i != 0) return APS_OK;
      aps_ctx* c = g->ctx[0];
      APS_CTX(c);
      if (F > 0) {
        for (int j = 1; j < N; ++j) {
          if (q_hi(j) == q_lo(j)) continue;
          APS_CUDA(cudaStreamWaitEvent(c->stream, g->ev[j][EV_SEARCH], 0));
          const size_t o = (size_t)q_lo(j) * 8;
          APS_CUDA(cudaMemcpyPeerAsync((char*)aps_gplan_records_device(plan[0]) + o, c->device,
                                       (const char*)aps_gplan_records_device(plan[j]) + o, g->ctx[j]->device,
                                       (size_t)(q_hi(j) - q_lo(j)) * 8, c->stream));
        }
        APS_TRY(record(g, 0, EV_GATHER));
        if (mutual) APS_TRY(aps_gplan_filter_mutual(plan[0]));
        APS_TRY(aps_gplan_compact(plan[0]));
      }
      APS_TRY(aps_gplan_download(plan[0], out));
      return F > 0 ? record(g, 0, EV_FINISH) : APS_OK;
    });
  drain(g);
  run_members(g, [&](int i) -> int {
    aps_gplan_destroy(plan[i]);
    return APS_OK;
  });
  if (rc != APS_OK && *out) {
    aps_matchlist_free(*out);
    *out = nullptr;
  }
  return rc;
}

// ------------------------------------------------------------------------------------------------
// featureMatchingPairwise across the members: member 0 uploads, the others copy its pooled matrix; member i matches the
// pairs whose column-major ordinal is congruent to i modulo N; the host lists are merged in cell order.
extern "C" int aps_group_feature_matching_pairwise(aps_group* g, const void* const* desc, const int64_t* counts, int n,
                                                   int D, int dtype, int layout, double match_threshold,
                                                   double max_ratio, int method, int64_t subset, uint64_t seed,
                                                   aps_matchlist** out) {
  if (!g || g->ctx.empty()) APS_FAIL(APS_ERR_NOGPU, "apsmatch:nogpu", "device group is NULL (no GPU context; there is no CPU path)");
  if (!out) APS_FAIL(APS_ERR_ARGS, "", "out is NULL");
  *out = nullptr;
  const int N = (int)g->ctx.size();
  std::fill(g->recorded.begin(), g->recorded.end(), 0);
  if (N == 1)
    return feature_matching_pairwise_impl(g->ctx[0], desc, counts, n, D, dtype, layout, match_threshold, max_ratio,
                                          method, subset, seed, 0, 1, out);
  if (n < 0 || (n > 0 && !counts)) APS_FAIL(APS_ERR_ARGS, "", "bad arguments");

  std::vector<aps_pplan*> plan((size_t)N, nullptr);
  std::vector<aps_matchlist*> part((size_t)N, nullptr);
  bool work = false;
  // 1: plans; member 0's host upload
  int rc = run_members(g, [&](int i) -> int {
    APS_TRY(aps_pplan_create(g->ctx[i], counts, n, D, dtype, &plan[i]));
    APS_TRY(aps_pplan_set_method(plan[i], method, subset, seed));
    if (i == 0) work = aps_pplan_total(plan[0]) > 0 && n >= 2;
    if (i != 0 || !work) return APS_OK;
    APS_TRY(record(g, 0, EV_START));
    APS_TRY(aps_pplan_upload(plan[0], desc, layout));
    return record(g, 0, EV_UPLOAD);
  });
  const size_t bytes = (size_t)(plan[0] ? aps_pplan_total(plan[0]) : 0) * D * (dtype == APS_F32 ? 4 : 1);
  // 2: the pooled raw matrix peer-to-peer to the other members
  if (rc == APS_OK && work)
    rc = run_members(g, [&](int i) -> int {
      aps_ctx* c = g->ctx[i];
      APS_CTX(c);
      if (i != 0) {
        APS_TRY(record(g, i, EV_START));
        APS_TRY(record(g, i, EV_UPLOAD));
        APS_CUDA(cudaStreamWaitEvent(c->stream, g->ev[0][EV_UPLOAD], 0));
        APS_CUDA(cudaMemcpyPeerAsync(aps_pplan_desc_device(plan[i]), c->device, aps_pplan_desc_device(plan[0]),
                                     g->ctx[0]->device, bytes, c->stream));
      }
      return record(g, i, EV_EXCHANGE);
    });
  // 3: K1 and this member's share of the pair list (member 0 leaves its matrix untouched until every copy is done)
  if (rc == APS_OK)
    rc = run_members(g, [&](int i) -> int {
      aps_ctx* c = g->ctx[i];
      APS_CTX(c);
      if (work) {
        if (i == 0)
          for (int j = 1; j < N; ++j) APS_CUDA(cudaStreamWaitEvent(c->stream, g->ev[j][EV_EXCHANGE], 0));
        APS_TRY(aps_pplan_prepare(plan[i]));
      }
      APS_TRY(aps_pplan_match(plan[i], match_threshold, max_ratio, i, N, &part[i]));
      return work ? record(g, i, EV_SEARCH) : APS_OK;
    });
  drain(g);
  run_members(g, [&](int i) -> int {
    aps_pplan_destroy(plan[i]);
    return APS_OK;
  });
  // 4: merge: pair o of the column-major list (cell i + j*n, i < j) comes from member o % N
  if (rc == APS_OK) {
    aps_matchlist* m = new (std::nothrow) aps_matchlist();
    if (!m) {
      aps_set_error(APS_ERR_ALLOC, "", "out of host memory");
      rc = APS_ERR_ALLOC;
    } else {
      m->n = n;
      m->has_metric = true;
      const size_t cells = (size_t)n * n;
      m->pair_ptr.assign(cells + 1, 0);
      int64_t total = 0;
      for (int r = 0; r < N; ++r) total += part[r]->total;
      m->rows.reserve((size_t)total * 2);
      m->metric.reserve((size_t)total);
      size_t o = 0;
      for (int j = 0; j < n; ++j)
        for (int i = 0; i < n; ++i) {
          const size_t cell = (size_t)i + (size_t)j * n;
          int64_t add = 0;
          if (i < j) {
            const aps_matchlist* src = part[o++ % (size_t)N];
            const int64_t a = src->pair_ptr[cell], b = src->pair_ptr[cell + 1];
            add = b - a;
            m->rows.insert(m->rows.end(), src->rows.begin() + 2 * a, src->rows.begin() + 2 * b);
            m->metric.insert(m->metric.end(), src->metric.begin() + a, src->metric.begin() + b);
          }
          m->pair_ptr[cell + 1] = m->pair_ptr[cell] + add;
        }
      m->total = m->pair_ptr[cells];
      *out = m;
    }
  }
  for (aps_matchlist* p : part) aps_matchlist_free(p);
  return rc;
}
