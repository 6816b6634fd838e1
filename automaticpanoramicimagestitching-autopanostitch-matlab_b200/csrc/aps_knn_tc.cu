// aps_knn_tc.cu -- K2: float nearest-neighbour CANDIDATE search on the 5th-gen tensor cores.
//
// Replaces the O(F^2 D) search behind  PP/mex/flann_knn.cpp:229-234 (global path) and the GEMM +
// two min passes of  PP/featureMatching/matchFeaturesScratch.m:351-358 (pairwise path) with
//     score(q, j) = (a_q . b_j) * scale_j + bias_j          (||a-b||^2 = ||a||^2 + ||b||^2 - 2 a.b)
// evaluated as a dense bf16 contraction: tcgen05.mma (cta_group::1, M=128, N=128, K=16 per
// instruction) with the accumulator in TMEM, operands staged in shared memory by TMA
// (SWIZZLE_128B, K-major), and a fused top-K' selection in the epilogue: the distance matrix is
// never written.  The K' best train rows per (query row, column segment) go to aps_rerank.cu, which
// recomputes them exactly in FP32 and proves the top-k complete.  K' = 8 for k <= 5; 6 when the operands are exact in
// bf16 (device flag, both variants launched, one exits at once); 16 for 6 <= k <= 12 (one variant, no exact-operand
// sub-variant: the proof keeps >= 4 ranks between the k-th neighbour and the list's floor, as K' = 8 keeps 3 for
// k = 5); 4 in the per-pair searches (k = 2) -- or, for
// per-pair sweeps of <= 48 tiles, the branch-free SEGMENT epilogue (KCT == 3, CS == 2; see top2_of_32 below):
// 16 epilogue warps, two sorted lists of three per row, no data-dependent branch.
//
// CTA = 384 threads (three warpgroups), persistent over work units.  A unit = TWO 128-row query blocks (256 rows, both A
// tiles resident in shared memory) x a range of 128-column train tiles; every B tile feeds two MMA
// groups (one per row block), which halves the operand traffic per output and lets each query row be
// owned by exactly ONE epilogue thread -- one top-K' list per row, half the insertions of a
// column-split epilogue.
//   warp 0   : TMA producer  (two A tiles per unit; per step one B tile, + per-column (scale,bias) on short sweeps)
//   warps 1-2: one single-thread tcgen05.mma issuer per row block (warp 1 also owns the TMEM allocation);
//              independent issuers remove head-of-line blocking between the two epilogue groups
//   warp 3   : idle (warpgroup 0 = the control warps: setmaxnreg.dec to 48 registers, setmaxnreg.inc to 224 for the
//              epilogue warpgroups, which no longer spill; 20 warps, 64 / 104 for the KCT == 3 variant)
//   warps 4-7: epilogue group 0 = row block 0, warps 8-11: group 1 = row block 1 (thread == query row,
//              tcgen05.ld 32x32b from the warp's TMEM lane quadrant).  Long sweeps (PRE), per 128-column tile:
//              (1) straight-line scan: tcgen05.ld .x32 double-buffered, 16 FMNMX3 trees = the maxima of the 16
//                  8-column groups of RAW accumulators, against a per-tile threshold derived from the row's K'-th
//                  best (theta) and the tile's (min,max) column scale / bias (aps_k_tile_bounds; the train view
//                  is sorted by scale so the bounds are tight) -- no per-column constant, no multiply;
//              (2) ONE warp vote; no lane flagged a group -> next tile (~270 instructions per tile and warp);
//              (3) otherwise the union of the flagged groups is RE-READ from TMEM (tcgen05.ld .x8, rounds of four)
//                  by the converged warp, the slot is handed back to the tensor pipe, and the flagged lanes scale,
//                  search and replace-min: scores in registers as packed keys (value bits & ~7 | slot), train-row
//                  indices in shared memory.  One run-time-indexed copy of the insertion code.  The column constants
//                  never cost an L2 round trip in the walk: every tile, each lane prefetches the NEXT tile's 4 scales
//                  (and biases) with one LDG.128 next to the tile-bounds prefetch; a flagged tile writes them once to
//                  the warp's 1 KB staging area (STS.128 per lane, in the (scale, bias) ring region that long sweeps do
//                  not use), and each round reads its groups' values with broadcast LDS.128 issued before the re-read.
//                  No per-tile wait on a constants ring either.
//              Short sweeps (!PRE: the lists never leave their filling phase) keep the per-chunk loop: scale every
//              32-column chunk, group maxima, branch-free replace-min for the groups that hold a candidate.
// TMEM: 4 accumulator slots of 128 columns = slot(tile parity, row block): the tensor pipe fills the
// slots of tile t+1 while both groups drain tile t.  Pipelines (all mbarrier based): B ring (4 x 32 KB),
// A pair (single buffered per unit), accumulator slots, (scale,bias) ring (short sweeps only).
// Scheduling: units that fill whole rounds of the grid span all train tiles; the last, partial round is
// balanced either by cutting its units into <= 4 equal column segments or by cutting its tile steps into
// one equal share per CTA (make_schedule), each piece filling its own candidate list of the row.
//
// What bounds it (C2 = 163840^2 pairs, D = 128; profiles/r2_ncu_history.txt, profiles/r2_ncu_k_knn_tc.txt):
//   * accumulators never read (-DAPS_TC_NOEPI): TMA + MMA alone 3.39 ms = 2027 TFLOP/s -- the floor of this tiling
//     (85 % of nominal; the same with the A operand in TMEM: shared-memory bandwidth is not the limiter);
//   * full kernel 4.35 ms = 1580 TFLOP/s = 0.98 of the measured cuBLAS bf16 burst figure (B200, 1000 W, 1965 MHz;
//     round 3: 4.60 ms, with the flagged groups' constants loaded from L2 in every round of the walk; round 2:
//     4.71-4.87 ms, before the register split; round 1: 5.79 ms; per-chunk group-gated version: 5.32 ms); C3 (F = 1e6,
//     long sweeps) 1635 TFLOP/s = 1.01 of it (round 2).
//     What is left at C2 is the epilogue's own work (per-tile clocks, -DAPS_TC_TILE_CLOCKS, profiles/tile_clocks.py):
//     1262 busy cycles per tile and warp on average against ~1200 for the MMAs; a tile with insertions (39 % of them)
//     takes ~2100 (of which ~910 insertions), one without ~730, and the epilogue warps still wait for acc_full 14 % of
//     their cycles.  K'(1 + ln(F/K')) ~ 67 insertions per row are inherent to a streaming top-K';
//   * not kept: A operand in TMEM with three slots (5.34 ms); separate scan / insert warps with setmaxnreg
//     (5.13 ms: the per-tile hand-off costs more than it frees); two lists per row on column halves with 16
//     epilogue warps (twice the insertions); fp16 accumulators (rounding breaks the completeness proof on
//     SIFT-like data: median d8-d4 gap 0.016);
//   * earlier designs: one row block per unit, epilogue split by columns, single MMA issuer: 8.23 ms; fully unrolled
//     register-resident sorted top-K: 348 KB of SASS, 69 % instruction-fetch stalls, 109 ms.
//
// Roofline: tensor pipe.  Algorithmic FLOPs = 2*D per (query, train) pair.  HBM traffic is
// negligible (operands stream from L2: every concurrently running CTA walks the same B tiles).
#include "aps_tc_ptx.cuh"

// the KCT == 3 instantiation leaves the unit loop before the streaming top-K' code ("loop is not reachable")
#pragma nv_diag_suppress 128

namespace {
using namespace aps_tc;

constexpr int TM = 128;        // query rows per MMA (UMMA M); a unit holds RB of these row blocks
constexpr int RB = 2;          // row blocks per unit == epilogue groups
constexpr int TN = 128;        // train rows per step (UMMA N)
constexpr int NUM_B_STAGES = 4;
constexpr int NUM_ACC_SLOTS = 2 * RB;  // slot = (tile parity) * RB + row block ; 4 x 128 columns = all of TMEM
constexpr int NUM_CS_STAGES = 8;
constexpr int KC = 8;          // candidates per (row, segment) for k <= 5
constexpr int KC_LARGE = 16;   // ... for 6 <= k <= 12
constexpr int CSPLIT = 1;      // epilogue groups per row block (each scans TN/CSPLIT columns of every tile, own list)
constexpr int MAX_SEG = 4 / CSPLIT;  // column segments of a tail unit; a row has MAX_SEG*CSPLIT <= 4 candidate lists
constexpr int NUM_EPI_WARPS = 4 * RB * CSPLIT;
// warpgroup 0: warp 0 producer, warps 1..RB MMA issuers (one per row block), warp 3 idle; the epilogue groups start
// at warpgroup 1, so that setmaxnreg (per warpgroup) can move registers from the control warps to the epilogue
constexpr int FIRST_EPI_WARP = 4;
static_assert(1 + RB <= FIRST_EPI_WARP, "producer and issuers fit in warpgroup 0");
constexpr int NUM_THREADS = 32 * (FIRST_EPI_WARP + NUM_EPI_WARPS);
static_assert(NUM_ACC_SLOTS * TN == 512, "TMEM budget");
// train-row slots per list in shared memory: KC for every list of up to KC candidates, one layout for all of them
__host__ __device__ constexpr int list_slots(int kct) { return kct > KC ? kct : KC; }

struct Barriers {
  uint64_t b_full[NUM_B_STAGES], b_empty[NUM_B_STAGES];
  uint64_t a_full, a_empty;
  uint64_t acc_full[NUM_ACC_SLOTS], acc_empty[NUM_ACC_SLOTS];
  uint64_t cs_full[NUM_CS_STAGES], cs_empty[NUM_CS_STAGES];
  uint32_t tmem_base;
  uint32_t pad;
};
// byte distance from a full barrier to its empty partner: one base register per ring, the partner is an immediate offset
constexpr uint32_t kAccEmptyOff = offsetof(Barriers, acc_empty) - offsetof(Barriers, acc_full);
constexpr uint32_t kCsEmptyOff = offsetof(Barriers, cs_empty) - offsetof(Barriers, cs_full);
// dynamic shared memory of a launch: A pair, B ring, (scale, bias) ring, the lists' train rows, barriers
constexpr size_t smem_bytes(int dp, int cs, int kct) {
  return 1024 + (size_t)RB * TM * dp * 2 + (size_t)NUM_B_STAGES * TN * dp * 2 + (size_t)NUM_CS_STAGES * 2 * TN * 4 +
         (size_t)RB * cs * list_slots(kct) * TM * 4 + sizeof(Barriers);
}
static_assert(smem_bytes(128, CSPLIT, KC_LARGE) <= 232448, "K' = 16 lists fit the 227 KB of a block at Dp = 128");

// The row's top-KC list lives in shared memory, slot-major ([slot][row], conflict-free), descending
// by score; addressed by 32-bit shared-window addresses (ld/st.shared, not generic).  Out of line
// on purpose (code size); returns the new K'-th best score.
__device__ __forceinline__ float4 lds_f32x4(uint32_t a) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
  return v;
}
__device__ __forceinline__ void sts_f32x4(uint32_t a, float4 v) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ uint32_t lds_u32(uint32_t a) { uint32_t v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
__device__ __forceinline__ void sts_u32(uint32_t a, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
constexpr uint32_t SLOT_STRIDE = TM * 4;                  // bytes between consecutive slots of one row

#ifdef APS_TC_TILE_CLOCKS
// Measurement aid (-DAPS_TC_TILE_CLOCKS, profiles/tile_clocks.py): lane 0 of every epilogue warp of a long-sweep launch
// writes one record of kClkWords words per tile: clock() cycles of (0) the acc_full wait, (1) the scan and vote, (2) the
// walk of the flagged groups without its insertions (per-tile staging, TMEM re-reads, waits for the column constants),
// (3) the insertions (search_group), (4) the whole tile; (5) the union of flagged groups, (6) the rounds, (7) flags
// (1: flagged, 2: partial tile, 4: first tile of the unit).  Records beyond kClkCap per warp are dropped; second-pass
// (nrows_dev) launches record nothing, so the buffer holds the last first-pass launch.
constexpr int kClkWords = 8, kClkCap = 8192, kClkCtas = 160;
__device__ uint32_t* g_tile_clk;    // [kClkCtas][8 epilogue warps][kClkCap][kClkWords]
__device__ uint32_t* g_tile_clk_n;  // [kClkCtas][8 epilogue warps] records of the last recorded launch
#define APS_CLK(...) __VA_ARGS__
#else
#define APS_CLK(...)
#endif

struct KParams {
  int64_t q0, q1, t0, t1;
  int dp;               // padded descriptor length (64 or 128)
  int nslot;            // candidate lists allocated per row (1..MAX_SEG)
  int units_full;       // units that span all tiles (list 0 only)
  int tail_units;       // row-block pairs of the last partial round ...
  int tail_seg;         // ... each split into this many column segments
  int64_t tile_lo;      // first TN-column tile (global tile grid)
  int64_t tile_hi;      // one past the last tile
  int tiles_per_seg;    // tiles per segment of a tail unit
  int tail_balanced;    // > 0: the tail's tile steps (tail_units x tiles, unit-major) are cut into `grid` equal
                        //    contiguous shares, one per CTA; value = pieces a share can consist of (2, or 3 when
                        //    the last full round is merged into the tail); <= nslot pieces per unit
  int grid;             // CTAs launched (balanced tail only)
  const float* colscale;  // [Ft_total + 256] per train row
  const float* colbias;   // [Ft_total + 256] per train row (read only by the BIAS variant)
  const float4* tile_bounds;  // per train tile: (1/scale_max, 1/scale_min, bias_max, -), 1e-6 safety included
  uint32_t* cand_idx;
  float* cand_score;
  float* dump;
  const aps_tc_unit* unit_table;  // batched (pairwise) mode: explicit units, one list per row; else nullptr
  int64_t n_table_units;
  int cand_stride;                // entries per list in cand_idx / cand_score (>= KCT; the rest is written empty)
  const int32_t* variant_flag;    // when set: this launch runs only if (*variant_flag != 0) == variant_want
  int variant_want;
  uint32_t idesc;                 // tcgen05 instruction descriptor (bf16 or fp16 operands, f32 accumulators)
  const int32_t* nrows_dev;       // second-pass mode: the query matrix holds *nrows_dev gathered rows (device-side
                                  // count); every unit is split into tail_seg column segments
};

struct Unit {
  int64_t qrow0;     // first query row (global) of the unit's 256-row block pair
  int64_t qend;      // rows >= qend are not the unit's (next image / end of range): computed, not stored
  int64_t t0, t1;    // train rows searched (columns outside are masked)
  int64_t out_row;   // candidate-buffer row of qrow0
  int64_t tl, th;    // tile range
  int seg;           // candidate list this unit fills
  int clear_from;    // this unit also marks the row's lists [clear_from, nslot) empty (nslot: none)
  bool skip;         // no work (balanced tail: a CTA's share may lie inside one unit)
};
__device__ __forceinline__ Unit get_unit(const KParams& P, int64_t u) {
  Unit x;
  if (P.unit_table) {
    const aps_tc_unit t = P.unit_table[u];
    x.qrow0 = t.qrow0; x.qend = t.qend; x.t0 = t.t0; x.t1 = t.t1; x.out_row = t.out_row;
    x.tl = t.t0 / TN; x.th = (t.t1 + TN - 1) / TN; x.seg = 0; x.clear_from = 1; x.skip = false;
    return x;
  }
  int64_t rb2;
  x.skip = false;
  if (u < P.units_full) {
    rb2 = u; x.tl = P.tile_lo; x.th = P.tile_hi; x.seg = 0; x.clear_from = CSPLIT;
  } else if (P.tail_balanced) {
    const int64_t v = u - P.units_full, G = P.grid;
    const int64_t j = v % G, k = v / G;  // CTA j's k-th piece (k < tail_balanced); units_full is a multiple of G
    const int64_t T = P.tile_hi - P.tile_lo, W = (int64_t)P.tail_units * T;
    const int64_t w0 = j * W / G, w1 = (j + 1) * W / G;
    const int64_t r0 = w0 / T, r = r0 + k;
    const int64_t a = (k == 0) ? w0 - r0 * T : 0;
    const int64_t b = min(T, w1 - r * T);
    x.skip = (w1 <= w0) || (b <= a);
    const int64_t own0 = ((r * T + 1) * G - 1) / W;  // CTA whose share holds the unit's first tile step
    const int64_t ownl = ((r * T + T) * G - 1) / W;  // ... and its last one
    x.seg = (int)(j - own0);
    x.clear_from = (x.seg == 0) ? (int)(ownl - own0 + 1) : P.nslot;
    rb2 = P.units_full + r;
    x.tl = P.tile_lo + a;
    x.th = P.tile_lo + b;
  } else {
    const int64_t v = u - P.units_full;
    x.seg = (int)(v / P.tail_units);                 // segment-major: neighbours share B tiles in L2
    rb2 = P.units_full + (v % P.tail_units);
    x.tl = P.tile_lo + (int64_t)x.seg * P.tiles_per_seg;
    x.th = min(P.tile_hi, x.tl + P.tiles_per_seg);
    x.clear_from = P.nslot;
  }
  x.qrow0 = P.q0 + rb2 * RB * TM; x.qend = P.q1; x.t0 = P.t0; x.t1 = P.t1; x.out_row = rb2 * RB * TM;
  return x;
}

// ---- branch-free selection for SHORT sweeps (per-pair searches, KCT == 3) -------------------------------------------
// A streaming top-K' with thread == query row makes a whole warp take the insert path whenever ANY of its 32 rows has a
// candidate in the chunk -- with only a few thousand columns per list that is nearly every chunk, and the ALU pipe
// (FMNMX / LOP3 / FSETP: one warp instruction per 2 cycles per SMSP) ends up 50 % busy at IPC 0.46 with two epilogue
// warps per SMSP (profiles/r1_ncu_k_knn_tc_pairwise.txt).  Here nothing depends on the data, so the columns of a tile
// can be split over CS = 2 epilogue groups per row block (4 warps per SMSP hide each other's latencies) without the
// doubled insertions that made the split lose in the streaming design: every score gets its column-in-tile packed
// into the 7 low mantissa bits (key; the 127-ulp truncation is inside the re-rank's eps), a min/max tree yields the two
// largest keys of each SEGMENT (the group's 64 columns of a tile), and those two are inserted into the group's sorted
// top-3 of the row (value + train row as payload).  Completeness (aps_rerank.cu, tile mode): a column outside a list is
// either one of its segment's two best (then it lost against the list's third entry) or is bounded by its segment's
// second best, which is itself below the third entry unless the list's two best share a segment (then W = the second).
__device__ __forceinline__ void top2_merge(float& h, float& l, const float h2, const float l2) {
  const float lo = fminf(h, h2);
  h = fmaxf(h, h2);
  l = fmaxf(fmaxf(lo, l), l2);
}
// top-2 keys of v[0..32): in place, result in (v[0], v[1])
__device__ __forceinline__ void top2_of_32(float (&v)[32]) {
#pragma unroll
  for (int i = 0; i < 32; i += 2) {
    const float a = v[i], b = v[i + 1];
    v[i] = fmaxf(a, b);
    v[i + 1] = fminf(a, b);
  }
#pragma unroll
  for (int st = 2; st < 32; st *= 2)
#pragma unroll
    for (int i = 0; i < 32; i += 2 * st) top2_merge(v[i], v[i + 1], v[i + st], v[i + st + 1]);
}
// insert (x, payload px) into the descending list (l1, l2, l3); strict '>' keeps the earlier entry first on ties
__device__ __forceinline__ void insert3(float x, uint32_t px, float& l1, float& l2, float& l3, uint32_t& p1, uint32_t& p2,
                                        uint32_t& p3) {
  const bool c1 = x > l1, c2 = x > l2, c3 = x > l3;
  l3 = c2 ? l2 : (c3 ? x : l3);
  p3 = c2 ? p2 : (c3 ? px : p3);
  l2 = c1 ? l1 : (c2 ? x : l2);
  p2 = c1 ? p1 : (c2 ? px : p2);
  l1 = c1 ? x : l1;
  p1 = c1 ? px : p1;
}
// minimum of a K' = 16 list (FMNMX3 tree)
__device__ __forceinline__ float list_min16(const float (&bv)[16]) {
  const float m0 = fminf(fminf(bv[0], bv[1]), bv[2]), m1 = fminf(fminf(bv[3], bv[4]), bv[5]);
  const float m2 = fminf(fminf(bv[6], bv[7]), bv[8]), m3 = fminf(fminf(bv[9], bv[10]), bv[11]);
  const float m4 = fminf(fminf(bv[12], bv[13]), bv[14]);
  return fminf(fminf(fminf(m0, m1), fminf(m2, m3)), fminf(m4, bv[15]));
}
constexpr uint32_t kKeyFloorBits = 0xff7fff80u;  // finite, below every real score: masked columns / empty entries
__host__ __device__ constexpr int threads_for(int cs) { return 32 * (FIRST_EPI_WARP + 4 * RB * cs); }
// Register split.  __launch_bounds__(threads, 1) makes ptxas allocate 65536 / threads registers per thread (rounded
// down to 8) at launch: 168 for 384 threads, 96 for 640.  Warpgroup 0 (mbarrier waits and address arithmetic) drops to
// kCtlRegs with setmaxnreg.dec; the epilogue warpgroups take what that frees with setmaxnreg.inc (224 and 104), so the
// per-tile scan and the insertion code no longer spill.  The launcher checks the allocation: setmaxnreg.inc would wait
// for ever if warpgroup 0 freed fewer registers than the epilogue asks for.
__host__ __device__ constexpr int ctl_regs(int cs) { return cs == 1 ? 48 : 64; }
__host__ __device__ constexpr int launch_regs(int cs) { return (65536 / threads_for(cs)) & ~7; }
__host__ __device__ constexpr int epi_regs(int cs) {
  return ((launch_regs(cs) * threads_for(cs) - 128 * ctl_regs(cs)) / (threads_for(cs) - 128)) & ~7;
}
static_assert(epi_regs(1) == 224 && epi_regs(2) == 104, "register split");

// KCT = candidates kept per list: 8, or 4 for the per-pair searches (k = 2: fewer insertions on short sweeps)
// CS = epilogue groups per row block (each scans TN/CS columns of every tile and keeps its own list)
template <bool BIAS, bool DUMP, bool PRE, int KCT, int CS = CSPLIT>
__global__ void __launch_bounds__(threads_for(CS), 1)
k_knn_tc(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_t, const KParams Pin) {
  // PRE runs only the long-sweep scan below, which reads the per-column constants from global memory: no ring stage
  static_assert(!PRE || (CS == 1 && !DUMP), "PRE has no (scale, bias) ring");
  // two launches cover one search when the list size depends on a device-side flag: the other one exits here
  if (Pin.variant_flag && ((*Pin.variant_flag != 0) != (Pin.variant_want != 0))) return;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // dynamic smem base is only guaranteed 16-byte aligned: align by hand
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  const int a_bytes = TM * Pin.dp * 2, b_bytes = TN * Pin.dp * 2;
  uint8_t* smem_a = smem;                                      // RB x a_bytes (both row blocks of the unit)
  uint8_t* smem_b = smem_a + RB * a_bytes;                     // NUM_B_STAGES x b_bytes
  float* smem_cs = (float*)(smem_b + NUM_B_STAGES * b_bytes);  // NUM_CS_STAGES x {TN scales, TN biases}
  constexpr int KL = list_slots(KCT);
  uint32_t* smem_topi = (uint32_t*)(smem_cs + NUM_CS_STAGES * 2 * TN);  // [RB*CS][KL][TM] train rows of the top-K'
  Barriers* bars = (Barriers*)(smem_topi + RB * CS * KL * TM);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ksl = Pin.dp / KSLAB;   // 128-byte K slabs per operand row
  const int kst = Pin.dp / 16;      // UMMA K steps per tile
  KParams P = Pin;
  if (P.nrows_dev) {  // device-side row count (rows gathered by aps_k_gather_rows): all units segmented
    const int64_t n = *P.nrows_dev;
    P.q1 = P.q0 + n;
    P.units_full = 0;
    P.tail_units = (int)((n + RB * TM - 1) / (RB * TM));
  }
  const int64_t num_units = P.unit_table ? P.n_table_units
                            : (P.tail_balanced ? (int64_t)P.units_full + (int64_t)P.tail_balanced * P.grid
                                               : (int64_t)P.units_full + (int64_t)P.tail_units * P.tail_seg);

  if (threadIdx.x == 0) {
    for (int i = 0; i < NUM_B_STAGES; ++i) { mbar_init(&bars->b_full[i], 1); mbar_init(&bars->b_empty[i], RB); }
    mbar_init(&bars->a_full, 1);
    mbar_init(&bars->a_empty, RB);
    for (int i = 0; i < NUM_ACC_SLOTS; ++i) { mbar_init(&bars->acc_full[i], 1); mbar_init(&bars->acc_empty[i], 4 * CS); }
    for (int i = 0; i < NUM_CS_STAGES; ++i) { mbar_init(&bars->cs_full[i], 1); mbar_init(&bars->cs_empty[i], (4 * RB * CS)); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {  // TMEM: all 512 columns (NUM_ACC_SLOTS x TN); one CTA per SM
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&bars->tmem_base)), "r"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = bars->tmem_base;

  // ptxas gives each role the register budget of the setmaxnreg that dominates it: the split sits inside the
  // role branches (a block reached from both sides gets the smaller budget), once per warpgroup
  if (warp < FIRST_EPI_WARP) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(ctl_regs(CS)));
    if (warp == 0) {
      // ===================================== TMA producer =====================================
      if (elect_one()) {
        uint32_t bs = 0, bph = 0, aph = 0, cs = 0, cph = 0;
        for (int64_t u = blockIdx.x; u < num_units; u += gridDim.x) {
          const Unit x = get_unit(P, u);
          if (x.tl >= x.th) continue;
          mbar_wait_backoff(&bars->a_empty, aph ^ 1);   // every MMA of the previous unit has read its A tiles
          mbar_arrive_expect_tx(&bars->a_full, (uint32_t)(RB * a_bytes));
          for (int r = 0; r < RB; ++r)
            for (int s = 0; s < ksl; ++s)
              tma_load_2d(smem_a + r * a_bytes + s * (TM * 128), &map_q, s * KSLAB,
                          (int)(x.qrow0 + r * TM), &bars->a_full);
          aph ^= 1;
          for (int64_t t = x.tl; t < x.th; ++t) {
            if constexpr (!PRE) {  // long sweeps read the per-column constants of the few candidate groups from L2
              mbar_wait_backoff(&bars->cs_empty[cs], cph ^ 1);
              mbar_arrive_expect_tx(&bars->cs_full[cs], (BIAS ? 2u : 1u) * TN * (uint32_t)sizeof(float));
              bulk_load_1d(smem_cs + cs * 2 * TN, P.colscale + t * TN, TN * (uint32_t)sizeof(float), &bars->cs_full[cs]);
              if (BIAS)
                bulk_load_1d(smem_cs + cs * 2 * TN + TN, P.colbias + t * TN, TN * (uint32_t)sizeof(float), &bars->cs_full[cs]);
              if (++cs == NUM_CS_STAGES) { cs = 0; cph ^= 1; }
            }
            mbar_wait_backoff(&bars->b_empty[bs], bph ^ 1);
            mbar_arrive_expect_tx(&bars->b_full[bs], (uint32_t)b_bytes);
            for (int s = 0; s < ksl; ++s)
              tma_load_2d(smem_b + bs * b_bytes + s * (TN * 128), &map_t, s * KSLAB, (int)(t * TN), &bars->b_full[bs]);
            if (++bs == NUM_B_STAGES) { bs = 0; bph ^= 1; }
          }
        }
      }
    } else if (warp <= RB) {
      // ===================================== MMA issuers =======================================
      // One issuing thread per row block: each waits only for ITS epilogue group's accumulator slot, so a
      // slow group (insertion-heavy tile) does not stall the other group's MMAs (no head-of-line blocking).
      if (elect_one()) {
        const int r = warp - 1;
        const uint32_t idesc = P.idesc;
        const uint32_t a_addr = smem_u32(smem_a + r * a_bytes);
        const uint32_t b_addr0 = smem_u32(smem_b);
        const uint32_t b_full0 = smem_u32(&bars->b_full[0]), b_empty0 = smem_u32(&bars->b_empty[0]);
        // this row block's accumulator slots are r (even tiles) and RB + r (odd tiles)
        const uint32_t acc_bar = smem_u32(&bars->acc_full[r]);
        uint32_t bs = 0, bph = 0, aph = 0, par = 0, acph = 0;  // par = tile parity, acph = its slot's phase
        for (int64_t u = blockIdx.x; u < num_units; u += gridDim.x) {
          const Unit x = get_unit(P, u);
          if (x.tl >= x.th) continue;
          mbar_wait(&bars->a_full, aph);
          aph ^= 1;
          for (uint32_t i = 0, n = (uint32_t)(x.th - x.tl); i < n; ++i) {
            mbar_wait(acc_bar + kAccEmptyOff + par * (RB * 8), acph ^ 1);
            mbar_wait(b_full0 + bs * 8, bph);
            tc_fence_after();
            const uint32_t b_addr = b_addr0 + bs * b_bytes;
            const uint32_t d_tmem = tmem_base + (par * RB + r) * TN;
            for (int k = 0; k < kst; ++k) {
              const int slab = k >> 2, kin = k & 3;  // 4 K steps (32 B each) per 128-byte swizzle row
              const uint64_t adesc = make_kmajor_sw128_desc(a_addr + slab * (TM * 128) + kin * 32);
              const uint64_t bdesc = make_kmajor_sw128_desc(b_addr + slab * (TN * 128) + kin * 32);
              umma_bf16(d_tmem, adesc, bdesc, idesc, k > 0 ? 1u : 0u);
            }
            tc_commit(acc_bar + par * (RB * 8));  // this row block's accumulator is ready for its epilogue group
            tc_commit(b_empty0 + bs * 8);           // B stage reusable once BOTH issuers' MMAs have read it (count RB)
            if (++bs == NUM_B_STAGES) { bs = 0; bph ^= 1; }
            par ^= 1;
            acph ^= par ^ 1;  // back to the even slot: next phase
          }
          tc_commit(&bars->a_empty);
        }
      }
    }  // warp 3: idle
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(epi_regs(CS)));
    // ===================================== epilogue =========================================
    // Group g (4 warps, one per TMEM lane quadrant) owns row block g of the unit: thread == query row.
    const int quad = warp & 3;        // TMEM lane quadrant this warp may access
    const int egrp = (warp - FIRST_EPI_WARP) >> 2;
    const int grp = egrp / CS;  // row block of the unit
    const int ch = egrp % CS;   // column part of every tile this warp scans
    constexpr int CG = TN / CS;
    const int row_in_tile = quad * 32 + lane;
    const uint32_t si = smem_u32(smem_topi + (egrp * KL) * TM + row_in_tile);  // this row's index slots
    // Position in the tile sequence (the MMA issuer's): accumulator slot (tile parity) * RB + grp and its phase, and
    // the (scale, bias) ring stage of short sweeps.  Barrier and TMEM addresses are 32-bit, computed once.
    const uint32_t acc_bar = smem_u32(&bars->acc_full[grp]), cs_bar = smem_u32(&bars->cs_full[0]);
    const uint32_t cs_smem0 = smem_u32(smem_cs + ch * CG);
    // long sweeps: the ring region holds one staging area per epilogue warp for the column constants of a flagged
    // tile (TN scales, TN biases: 8 warps x 1 KB = the ring's 8 KB)
    static_assert(NUM_EPI_WARPS * 2 * TN <= NUM_CS_STAGES * 2 * TN, "staging fits in the (scale, bias) ring");
    const uint32_t stage = smem_u32(smem_cs) + (warp - FIRST_EPI_WARP) * (2 * TN * 4);
    const uint32_t tmem_row = tmem_base + ((uint32_t)(quad * 32) << 16) + grp * TN + ch * CG;
    uint32_t par = 0, acph = 0, cs = 0, cph = 0;
    APS_CLK(uint32_t clk_n = 0;)
    auto next_tile = [&]() {
      par ^= 1;
      acph ^= par ^ 1;
      if (!PRE && ++cs == NUM_CS_STAGES) { cs = 0; cph ^= 1; }
    };
    for (int64_t u = blockIdx.x; u < num_units; u += gridDim.x) {
      const Unit x = get_unit(P, u);
      if (x.skip) continue;  // balanced tail: this CTA's share has no second piece
      const int64_t qrow = x.qrow0 + grp * TM + row_in_tile;
      // train columns are 32-bit (cand_idx): tile loops count and compare in 32 bits.  A column segment can start past
      // the last tile (tl > th: e.g. 5 tiles in 4 segments of 2): no tiles, but its lists are still written empty.
      const uint32_t nt = x.th > x.tl ? (uint32_t)(x.th - x.tl) : 0u, ct0 = (uint32_t)x.t0, ct1 = (uint32_t)x.t1;
      if constexpr (KCT == 3) {
        // ---- short sweeps: branch-free two-best per segment, merged into the group's sorted top-3 of the row ----
        float l1 = __uint_as_float(kKeyFloorBits), l2 = l1, l3 = l1;
        uint32_t p1 = 0xffffffffu, p2 = 0xffffffffu, p3 = 0xffffffffu;
        uint32_t col0 = (uint32_t)(x.tl * TN) + ch * CG;
        for (uint32_t i = 0; i < nt; ++i, col0 += TN, next_tile()) {
          mbar_wait(acc_bar + par * (RB * 8), acph);
          mbar_wait(cs_bar + cs * 8, cph);
          tc_fence_after();
          const uint32_t cscale = cs_smem0 + cs * (2 * TN * 4);
          const bool partial = (col0 < ct0) || (col0 + CG > ct1);
          const uint32_t taddr = tmem_row + par * (RB * TN);
          float m1 = __uint_as_float(kKeyFloorBits), m2 = m1;
#pragma unroll 1
          for (int c = 0; c < CG / 32; ++c) {
            float cur[32];
            tmem_ld32(taddr + c * 32, cur);  // the other warps of the sub-partition hide this latency
            tmem_wait_ld(cur);
#pragma unroll
            for (int g = 0; g < 4; ++g) {
              const float4 s0 = lds_f32x4(cscale + (c * 32 + 8 * g) * 4);
              const float4 s1 = lds_f32x4(cscale + (c * 32 + 8 * g + 4) * 4);
              if (BIAS) {
                const float4 b0 = lds_f32x4(cscale + (TN + c * 32 + 8 * g) * 4);
                const float4 b1 = lds_f32x4(cscale + (TN + c * 32 + 8 * g + 4) * 4);
                cur[8 * g + 0] = fmaf(cur[8 * g + 0], s0.x, b0.x); cur[8 * g + 1] = fmaf(cur[8 * g + 1], s0.y, b0.y);
                cur[8 * g + 2] = fmaf(cur[8 * g + 2], s0.z, b0.z); cur[8 * g + 3] = fmaf(cur[8 * g + 3], s0.w, b0.w);
                cur[8 * g + 4] = fmaf(cur[8 * g + 4], s1.x, b1.x); cur[8 * g + 5] = fmaf(cur[8 * g + 5], s1.y, b1.y);
                cur[8 * g + 6] = fmaf(cur[8 * g + 6], s1.z, b1.z); cur[8 * g + 7] = fmaf(cur[8 * g + 7], s1.w, b1.w);
              } else {
                cur[8 * g + 0] *= s0.x; cur[8 * g + 1] *= s0.y; cur[8 * g + 2] *= s0.z; cur[8 * g + 3] *= s0.w;
                cur[8 * g + 4] *= s1.x; cur[8 * g + 5] *= s1.y; cur[8 * g + 6] *= s1.z; cur[8 * g + 7] *= s1.w;
              }
            }
            const uint32_t cbase = (uint32_t)(ch * CG + c * 32);  // column-in-tile of cur[0]
#pragma unroll
            for (int j = 0; j < 32; ++j)  // key = score with the column-in-tile in the 7 low mantissa bits
              cur[j] = __uint_as_float((__float_as_uint(cur[j]) & ~127u) | (cbase + (uint32_t)j));
            if (partial) {  // first / last tile of the train image: foreign columns can never be selected
              const int lo = max((int)(ct0 - col0), 0) - c * 32, hi = min((int)(ct1 - col0), CG) - c * 32;
#pragma unroll
              for (int j = 0; j < 32; ++j)
                if (j < lo || j >= hi) cur[j] = __uint_as_float(kKeyFloorBits | (cbase + (uint32_t)j));
            }
            top2_of_32(cur);
            top2_merge(m1, m2, cur[0], cur[1]);
          }
          tc_fence_before();
          __syncwarp();
          if (lane == 0) {
            mbar_arrive(acc_bar + kAccEmptyOff + par * (RB * 8));
            mbar_arrive(cs_bar + kCsEmptyOff + cs * 8);
          }
          const uint32_t base = col0 - ch * CG;
          insert3(m1, base + (__float_as_uint(m1) & 127u), l1, l2, l3, p1, p2, p3);
          insert3(m2, base + (__float_as_uint(m2) & 127u), l1, l2, l3, p1, p2, p3);
        }
        if (qrow < x.qend) {  // CS lists of 3 per row, packed: [row][ch][3]
          const int64_t o = (x.out_row + grp * TM + row_in_tile) * P.cand_stride + ch * 3;
          const float floor_v = -1.0e38f;  // entries that never left the floor: fewer than 3 selectable columns
          P.cand_idx[o + 0] = l1 > floor_v ? p1 : 0xffffffffu; P.cand_score[o + 0] = l1 > floor_v ? l1 : -CUDART_INF_F;
          P.cand_idx[o + 1] = l2 > floor_v ? p2 : 0xffffffffu; P.cand_score[o + 1] = l2 > floor_v ? l2 : -CUDART_INF_F;
          P.cand_idx[o + 2] = l3 > floor_v ? p3 : 0xffffffffu; P.cand_score[o + 2] = l3 > floor_v ? l3 : -CUDART_INF_F;
        }
        continue;
      }
      // row-private top-KC (unsorted; aps_rerank.cu orders exactly): scores in registers, train rows in smem.  The low
      // mantissa bits of a retained score hold its slot number: 3 bits, 4 for K' = 16
      constexpr uint32_t kSlot = KCT > 8 ? 15u : 7u;
      float bv[KCT];
#pragma unroll
      for (int i = 0; i < KCT; ++i) {
        bv[i] = __uint_as_float((0xff7fffffu & ~kSlot) | (uint32_t)i);  // ~ -FLT_MAX with the slot number in the low bits
        sts_u32(si + i * SLOT_STRIDE, 0xffffffffu);
      }
      float theta = bv[KCT - 1];    // min of bv == the row's K'-th best score so far (empty slots: -FLT_MAX)
      int minpos = KCT - 1;         // slot holding it
      const float4* tbp = P.tile_bounds + x.tl;
      float4 tb_next = (PRE && nt > 0) ? __ldg(tbp) : make_float4(0.f, 0.f, 0.f, 0.f);
      uint32_t col0 = (uint32_t)(x.tl * TN) + ch * CG;
      // long sweeps: the tile's column constants, lane l holding columns 4l .. 4l+3, loaded one tile ahead
      float4 cs_next = make_float4(0.f, 0.f, 0.f, 0.f), cb_next = cs_next;
      if (PRE && nt > 0) {
        cs_next = __ldg(reinterpret_cast<const float4*>(P.colscale + col0) + lane);
        if (BIAS) cb_next = __ldg(reinterpret_cast<const float4*>(P.colbias + col0) + lane);
      }
      for (uint32_t i = 0; i < nt; ++i, col0 += TN, next_tile()) {
        const uint32_t acc_off = par * (RB * 8);
        // (clk_meta: flags | union << 8 | rounds << 16)
        APS_CLK(const uint32_t ck0 = (uint32_t)clock(); uint32_t ck_vote = 0, ck_walk = 0, ck_ins = 0,
                clk_meta = i == 0 ? 4u : 0u;)
        mbar_wait(acc_bar + acc_off, acph);
        if (!PRE) mbar_wait(cs_bar + cs * 8, cph);
        tc_fence_after();
        APS_CLK(const uint32_t ck1 = (uint32_t)clock();)
        const uint32_t cscale = cs_smem0 + cs * (2 * TN * 4);
        const bool partial = (col0 < ct0) || (col0 + CG > ct1);
        const uint32_t taddr = tmem_row + par * (RB * TN);
        // Conservative pre-filter on the RAW accumulators: a column can only beat theta if
        //   acc > (theta - bias_max(tile)) / scale_max(tile)     (1/scale_min when the numerator is negative);
        // train rows are sorted by scale (aps_prep.cu), so the bound is tight and the common path needs
        // neither the per-column constants nor a multiply.
        const float4 tb = tb_next;  // fetched one tile ahead: the global-load latency stays off the critical path
        const float4 cs_cur = cs_next, cb_cur = cb_next;  // (same)
        if (PRE && i + 1 < nt) {
          tb_next = __ldg(tbp + i + 1);
          cs_next = __ldg(reinterpret_cast<const float4*>(P.colscale + col0 + TN) + lane);
          if (BIAS) cb_next = __ldg(reinterpret_cast<const float4*>(P.colbias + col0 + TN) + lane);
        }
        auto pre_threshold = [&](float th) {
          const float num = th - tb.z - 1.0e-6f * (fabsf(th) + fabsf(tb.z));
          return num * (num >= 0.f ? tb.x : tb.y);
        };
        float thr_pre = PRE ? pre_threshold(theta) : 0.f;
        float va[32], vb[32];
        bool slot_released = false;  // (warp-uniform)
        if constexpr (PRE && CS == 1 && !DUMP) {
          // ---- long sweeps: straight-line scan of the whole tile, candidates re-read from TMEM ----
          // (1) the 16 group maxima of the row's 128 raw accumulators (FMNMX3 trees, no branch, no per-column constant);
          // (2) ONE warp vote per tile: no lane can hold a candidate -> next tile (about half of the tiles of C2, most
          //     of the tiles of longer sweeps);
          // (3) otherwise the union of the lanes' candidate groups is walked by the converged warp: the group's 8
          //     accumulators are re-read from TMEM (tcgen05.ld .x8 -- the tensor pipe does not touch the slot before
          //     acc_empty), scaled and searched by the lanes that flagged it.  One copy of the insertion code, indexed
          //     at run time, instead of one per (chunk, group): the scan stays in the instruction cache fully unrolled.
          // The lists are the ones the per-chunk loop below builds: same order of columns, same exact test against
          // theta; only the conservative raw gate is evaluated once per tile instead of once per chunk.
#ifndef APS_TC_NOEPI   // (measurement aid: -DAPS_TC_NOEPI leaves the accumulators unread = the TMA + MMA floor)
          float rm[16];
          tmem_ld32(taddr, va);
          tmem_wait_ld(va);
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            float(&cur)[32] = (c & 1) ? vb : va;
            float(&nxt)[32] = (c & 1) ? va : vb;
            if (c + 1 < 4) tmem_ld32(taddr + (c + 1) * 32, nxt);
#pragma unroll
            for (int g = 0; g < 4; ++g) {
              float m = fmaxf(fmaxf(cur[8 * g], cur[8 * g + 1]), cur[8 * g + 2]);
              m = fmaxf(fmaxf(m, cur[8 * g + 3]), cur[8 * g + 4]);
              m = fmaxf(fmaxf(m, cur[8 * g + 5]), cur[8 * g + 6]);
              rm[4 * c + g] = fmaxf(m, cur[8 * g + 7]);
            }
            if (c + 1 < 4) tmem_wait_ld(nxt);
          }
          float tmax = fmaxf(fmaxf(rm[0], rm[1]), rm[2]);
#pragma unroll
          for (int g = 3; g < 15; g += 2) tmax = fmaxf(fmaxf(tmax, rm[g]), rm[g + 1]);
          tmax = fmaxf(tmax, rm[15]);
          const bool flagged = __any_sync(0xffffffffu, partial || tmax > thr_pre);
          APS_CLK(ck_vote = (uint32_t)clock(); clk_meta |= (flagged ? 1u : 0u) | (__any_sync(~0u, partial) ? 2u : 0u);)
          if (flagged) {
            uint32_t pend = 0;
#pragma unroll
            for (int g = 0; g < 16; ++g) pend |= (rm[g] > thr_pre) ? (1u << g) : 0u;
            if (partial) pend = 0xffffu;
            uint32_t uni = __reduce_or_sync(0xffffffffu, pend);
            // the tile's constants, prefetched a tile ahead, go to this warp's staging area once (one STS.128 per
            // lane); every round then reads its groups' 8 values with broadcast LDS.128: no L2 round trip in the walk
            sts_f32x4(stage + 16 * lane, cs_cur);
            if (BIAS) sts_f32x4(stage + TN * 4 + 16 * lane, cb_cur);
            __syncwarp();
            APS_CLK(clk_meta |= (uint32_t)__popc(uni) << 8;)
            // one flagged group of this lane: scale, mask, insert (inlined once per stash position below)
            auto search_group = [&](float(&v)[8], const int g, const float4 (&s)[2], const float4 (&b)[2]) {
              const float4 s0 = s[0], s1 = s[1];
              if (BIAS) {
                const float4 b0 = b[0], b1 = b[1];
                v[0] = fmaf(v[0], s0.x, b0.x); v[1] = fmaf(v[1], s0.y, b0.y);
                v[2] = fmaf(v[2], s0.z, b0.z); v[3] = fmaf(v[3], s0.w, b0.w);
                v[4] = fmaf(v[4], s1.x, b1.x); v[5] = fmaf(v[5], s1.y, b1.y);
                v[6] = fmaf(v[6], s1.z, b1.z); v[7] = fmaf(v[7], s1.w, b1.w);
              } else {
                v[0] *= s0.x; v[1] *= s0.y; v[2] *= s0.z; v[3] *= s0.w;
                v[4] *= s1.x; v[5] *= s1.y; v[6] *= s1.z; v[7] *= s1.w;
              }
              if (partial) {  // first / last tile of the searched range: foreign columns can never be selected
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                  const uint32_t col = col0 + 8 * g + j;
                  if (col < ct0 || col >= ct1) v[j] = -CUDART_INF_F;
                }
              }
              float gm = fmaxf(fmaxf(v[0], v[1]), v[2]);
              gm = fmaxf(fmaxf(gm, v[3]), v[4]);
              gm = fmaxf(fmaxf(gm, v[5]), v[6]);
              gm = fmaxf(gm, v[7]);
              while (gm > theta) {  // loops only if the same 8 columns hold a second candidate
                int js = 7;
#pragma unroll
                for (int j = 6; j >= 0; --j) js = (v[j] == gm) ? j : js;
                sts_u32(si + minpos * SLOT_STRIDE, col0 + 8 * g + js);
                const float key = __uint_as_float((__float_as_uint(gm) & ~kSlot) | (uint32_t)minpos);
#pragma unroll
                for (int k = 0; k < KCT; ++k) bv[k] = (k == minpos) ? key : bv[k];
                if constexpr (KCT == 16) {
                  theta = list_min16(bv);
                } else if constexpr (KCT == 8) {
                  float m01 = fminf(fminf(bv[0], bv[1]), bv[2]);
                  float m23 = fminf(fminf(bv[3], bv[4]), bv[5]);
                  theta = fminf(fminf(m01, m23), fminf(bv[6], bv[7]));
                } else if constexpr (KCT == 6) {
                  theta = fminf(fminf(fminf(bv[0], bv[1]), bv[2]), fminf(fminf(bv[3], bv[4]), bv[5]));
                } else {
                  theta = fminf(fminf(bv[0], bv[1]), fminf(bv[2], bv[3]));
                }
                minpos = (int)(__float_as_uint(theta) & kSlot);
#pragma unroll
                for (int j = 0; j < 8; ++j) v[j] = (j == js) ? -CUDART_INF_F : v[j];
                gm = fmaxf(fmaxf(v[0], v[1]), v[2]);
                gm = fmaxf(fmaxf(gm, v[3]), v[4]);
                gm = fmaxf(fmaxf(gm, v[5]), v[6]);
                gm = fmaxf(gm, v[7]);
              }
            };
            // Rounds of up to four flagged groups: their accumulators are copied out of TMEM first and, once nothing is
            // left to read, the slot goes back to the tensor pipe BEFORE the insertions run -- a tile with candidates
            // (the slow 40 %) no longer holds up the MMAs of the tile after next.
            while (uni) {
              int gq[4];
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                gq[q] = uni ? __ffs((int)uni) - 1 : 31;  // 31: no group (bit 31 of pend is never set)
                uni &= uni - 1;
              }
              // the groups' scales (and biases) from the staging area, in flight together with the TMEM re-read (same
              // address in every lane: a broadcast)
              float4 gs[4][2], gb[4][2];
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                const uint32_t s4 = stage + 32 * (gq[q] & 15);
                gs[q][0] = lds_f32x4(s4);
                gs[q][1] = lds_f32x4(s4 + 16);
                if (BIAS) {
                  gb[q][0] = lds_f32x4(s4 + TN * 4);
                  gb[q][1] = lds_f32x4(s4 + TN * 4 + 16);
                }
              }
              float vs[32];
              __syncwarp();
#pragma unroll
              for (int q = 0; q < 4; ++q) tmem_ld8(taddr + 8 * (gq[q] & 15), *reinterpret_cast<float(*)[8]>(vs + 8 * q));
              tmem_wait_ld(vs);
#ifdef APS_TC_TILE_CLOCKS
              {  // consume every constant here, so that the wait for them is counted in the walk, not the insertions
                float w = 0.f;
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                  asm volatile("add.f32 %0, %0, %1;" : "+f"(w) : "f"(gs[q][0].x + gs[q][0].y + gs[q][0].z + gs[q][0].w));
                  asm volatile("add.f32 %0, %0, %1;" : "+f"(w) : "f"(gs[q][1].x + gs[q][1].y + gs[q][1].z + gs[q][1].w));
                  if (BIAS) {
                    asm volatile("add.f32 %0, %0, %1;" : "+f"(w) : "f"(gb[q][0].x + gb[q][0].y + gb[q][0].z + gb[q][0].w));
                    asm volatile("add.f32 %0, %0, %1;" : "+f"(w) : "f"(gb[q][1].x + gb[q][1].y + gb[q][1].z + gb[q][1].w));
                  }
                }
                clk_meta |= (__float_as_uint(w) == 0x7fc00001u) ? 8u : 0u;
              }
#endif
              if (uni == 0u) {
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(acc_bar + kAccEmptyOff + acc_off);
                slot_released = true;
              }
              APS_CLK(clk_meta += 1u << 16; const uint32_t cr = (uint32_t)clock();)
#pragma unroll
              for (int q = 0; q < 4; ++q)
                if ((pend >> gq[q]) & 1u) search_group(*reinterpret_cast<float(*)[8]>(vs + 8 * q), gq[q], gs[q], gb[q]);
              APS_CLK(__syncwarp(); ck_ins += (uint32_t)clock() - cr;)
            }
            APS_CLK(ck_walk = (uint32_t)clock() - ck_vote - ck_ins;)
          }
#endif
        } else {
        if (CS == 1) {  // two warps per sub-partition: double-buffer the TMEM loads
          tmem_ld32(taddr, va);
          tmem_wait_ld(va);
        }
#pragma unroll 1
        for (int c2 = 0; c2 < CG / 64 + (CG % 64 ? 1 : 0); ++c2) {
#pragma unroll
          for (int h = 0; h < (CG >= 64 ? 2 : 1); ++h) {
            const int c = 2 * c2 + h;
            float(&cur)[32] = (CS == 1 && h) ? vb : va;
            float(&nxt)[32] = (CS == 1 && h) ? va : vb;
            if (CS == 1) {
              if (c + 1 < CG / 32) tmem_ld32(taddr + (c + 1) * 32, nxt);
            } else {  // four warps per sub-partition hide the load latency of each other: single buffer
              tmem_ld32(taddr + c * 32, cur);
              tmem_wait_ld(cur);
            }
            float rm[4] = {0.f, 0.f, 0.f, 0.f};
            if (PRE) {
#pragma unroll
              for (int g = 0; g < 4; ++g) {
                float m = fmaxf(fmaxf(cur[8 * g], cur[8 * g + 1]), cur[8 * g + 2]);
                m = fmaxf(fmaxf(m, cur[8 * g + 3]), cur[8 * g + 4]);
                m = fmaxf(fmaxf(m, cur[8 * g + 5]), cur[8 * g + 6]);
                rm[g] = fmaxf(m, cur[8 * g + 7]);
              }
            }
            // PRE = false (short units, e.g. one image pair: the lists never leave their filling phase, the
            // pre-filter would reject almost nothing) goes straight to the scaled scores
            const bool gate_all = !PRE || partial || DUMP;
            if (gate_all || fmaxf(fmaxf(rm[0], rm[1]), fmaxf(rm[2], rm[3])) > thr_pre) {
              // group-gated slow path: only the 8-column groups whose raw maximum can hold a candidate are scaled and
              // searched (in the middle of a sweep that is usually one group of the chunk, not four)
              bool inserted = false;
#pragma unroll
              for (int g = 0; g < 4; ++g) {
                if (gate_all || rm[g] > thr_pre) {
                  const float4 s0 = lds_f32x4(cscale + (c * 32 + 8 * g) * 4);
                  const float4 s1 = lds_f32x4(cscale + (c * 32 + 8 * g + 4) * 4);
                  if (BIAS) {
                    const float4 b0 = lds_f32x4(cscale + (TN + c * 32 + 8 * g) * 4);
                    const float4 b1 = lds_f32x4(cscale + (TN + c * 32 + 8 * g + 4) * 4);
                    cur[8 * g + 0] = fmaf(cur[8 * g + 0], s0.x, b0.x); cur[8 * g + 1] = fmaf(cur[8 * g + 1], s0.y, b0.y);
                    cur[8 * g + 2] = fmaf(cur[8 * g + 2], s0.z, b0.z); cur[8 * g + 3] = fmaf(cur[8 * g + 3], s0.w, b0.w);
                    cur[8 * g + 4] = fmaf(cur[8 * g + 4], s1.x, b1.x); cur[8 * g + 5] = fmaf(cur[8 * g + 5], s1.y, b1.y);
                    cur[8 * g + 6] = fmaf(cur[8 * g + 6], s1.z, b1.z); cur[8 * g + 7] = fmaf(cur[8 * g + 7], s1.w, b1.w);
                  } else {
                    cur[8 * g + 0] *= s0.x; cur[8 * g + 1] *= s0.y; cur[8 * g + 2] *= s0.z; cur[8 * g + 3] *= s0.w;
                    cur[8 * g + 4] *= s1.x; cur[8 * g + 5] *= s1.y; cur[8 * g + 6] *= s1.z; cur[8 * g + 7] *= s1.w;
                  }
                  if (partial || DUMP) {  // first / last tile of the searched range: mask foreign columns
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                      const int64_t col = col0 + c * 32 + 8 * g + j;
                      const bool ok = col >= x.t0 && col < x.t1;
                      if (DUMP && ok && qrow < P.q1) P.dump[(qrow - P.q0) * (P.t1 - P.t0) + (col - P.t0)] = cur[8 * g + j];
                      if (!ok) cur[8 * g + j] = -CUDART_INF_F;
                    }
                  }
                  float gm = fmaxf(fmaxf(cur[8 * g], cur[8 * g + 1]), cur[8 * g + 2]);
                  gm = fmaxf(fmaxf(gm, cur[8 * g + 3]), cur[8 * g + 4]);
                  gm = fmaxf(fmaxf(gm, cur[8 * g + 5]), cur[8 * g + 6]);
                  gm = fmaxf(gm, cur[8 * g + 7]);
                  // branch-free replace-min of the group's maximum; loops only if the same 8 columns hold
                  // a second candidate
                  while (gm > theta) {
                    inserted = true;
                    int js = 7;
#pragma unroll
                    for (int j = 6; j >= 0; --j) js = (cur[8 * g + j] == gm) ? j : js;
                    sts_u32(si + minpos * SLOT_STRIDE, (uint32_t)(col0 + c * 32 + 8 * g + js));
                    // the 3 (K' = 16: 4) low mantissa bits of a retained score hold its slot number: one FMNMX tree
                    // yields the new minimum AND its slot (the 7- or 15-ulp truncation is covered by the re-rank's eps)
                    const float key = __uint_as_float((__float_as_uint(gm) & ~kSlot) | (uint32_t)minpos);
#pragma unroll
                    for (int i = 0; i < KCT; ++i) bv[i] = (i == minpos) ? key : bv[i];
                    if constexpr (KCT == 16) {
                      theta = list_min16(bv);
                    } else if constexpr (KCT == 8) {
                      float m01 = fminf(fminf(bv[0], bv[1]), bv[2]);
                      float m23 = fminf(fminf(bv[3], bv[4]), bv[5]);
                      theta = fminf(fminf(m01, m23), fminf(bv[6], bv[7]));
                    } else if constexpr (KCT == 6) {
                      theta = fminf(fminf(fminf(bv[0], bv[1]), bv[2]), fminf(fminf(bv[3], bv[4]), bv[5]));
                    } else if constexpr (KCT == 4) {
                      theta = fminf(fminf(bv[0], bv[1]), fminf(bv[2], bv[3]));
                    } else {
                      theta = fminf(fminf(bv[0], bv[1]), bv[2]);  // (KCT == 3 never reaches the streaming path)
                    }
                    minpos = (int)(__float_as_uint(theta) & kSlot);
#pragma unroll
                    for (int j = 0; j < 8; ++j) cur[8 * g + j] = (j == js) ? -CUDART_INF_F : cur[8 * g + j];
                    gm = fmaxf(fmaxf(cur[8 * g], cur[8 * g + 1]), cur[8 * g + 2]);
                    gm = fmaxf(fmaxf(gm, cur[8 * g + 3]), cur[8 * g + 4]);
                    gm = fmaxf(fmaxf(gm, cur[8 * g + 5]), cur[8 * g + 6]);
                    gm = fmaxf(gm, cur[8 * g + 7]);
                  }
                }
              }
              if (PRE && inserted) thr_pre = pre_threshold(theta);
            }
            if (CS == 1 && c + 1 < CG / 32) tmem_wait_ld(nxt);
          }
        }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (!slot_released) mbar_arrive(acc_bar + kAccEmptyOff + acc_off);
          if (!PRE) mbar_arrive(cs_bar + kCsEmptyOff + cs * 8);
        }
#ifdef APS_TC_TILE_CLOCKS
        if (PRE && g_tile_clk && !P.nrows_dev && blockIdx.x < kClkCtas && lane == 0) {
          const uint32_t ck2 = (uint32_t)clock(), w = blockIdx.x * NUM_EPI_WARPS + (warp - FIRST_EPI_WARP);
          if (clk_n < (uint32_t)kClkCap) {
            uint4* r = reinterpret_cast<uint4*>(g_tile_clk + ((size_t)w * kClkCap + clk_n) * kClkWords);
            r[0] = make_uint4(ck1 - ck0, ck_vote - ck1, ck_walk, ck_ins);
            r[1] = make_uint4(ck2 - ck0, (clk_meta >> 8) & 0xffu, clk_meta >> 16, clk_meta & 0xffu);
          }
          g_tile_clk_n[w] = min(++clk_n, (uint32_t)kClkCap);
        }
#endif
      }
      if (qrow < x.qend) {
        const int cstr = P.cand_stride;
        const int64_t o = ((x.out_row + grp * TM + row_in_tile) * P.nslot + x.seg * CS + ch) * cstr;
#pragma unroll
        for (int i = 0; i < KCT; ++i) {
          P.cand_idx[o + i] = lds_u32(si + i * SLOT_STRIDE);
          P.cand_score[o + i] = bv[i];
        }
        for (int i = KCT; i < cstr; ++i) {
          P.cand_idx[o + i] = 0xffffffffu;
          P.cand_score[o + i] = -CUDART_INF_F;
        }
        if (ch == 0)  // e.g. rows of full-width units use the first CS lists: mark the others empty
          for (int sl = x.clear_from - x.seg * CS; sl < P.nslot - x.seg * CS; ++sl)
            for (int i = 0; i < cstr; ++i) {
              P.cand_idx[o + sl * cstr + i] = 0xffffffffu;
              P.cand_score[o + sl * cstr + i] = -CUDART_INF_F;
            }
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

}  // namespace

#ifdef APS_TC_TILE_CLOCKS
// op 0: allocate (once) and zero the record buffer and point the kernel at it; op 1: copy the counts
// ([kClkCtas * 8] uint32) and the records ([kClkCtas * 8 * kClkCap * kClkWords] uint32) to host memory;
// op 2: write (kClkCtas, epilogue warps, kClkCap, kClkWords) to counts.  Not part of apsmatch.h.
extern "C" __attribute__((visibility("default"))) int aps_debug_tile_clocks(int op, uint32_t* counts, uint32_t* records) {
  static uint32_t *d_rec = nullptr, *d_n = nullptr;
  const size_t nw = (size_t)kClkCtas * NUM_EPI_WARPS, nrec = nw * kClkCap * kClkWords;
  if (op == 2) {
    counts[0] = kClkCtas; counts[1] = NUM_EPI_WARPS; counts[2] = kClkCap; counts[3] = kClkWords;
    return APS_OK;
  }
  if (op == 0) {
    if (!d_rec) {
      APS_CUDA(cudaMalloc((void**)&d_rec, nrec * 4));
      APS_CUDA(cudaMalloc((void**)&d_n, nw * 4));
      APS_CUDA(cudaMemcpyToSymbol(g_tile_clk, &d_rec, sizeof d_rec));
      APS_CUDA(cudaMemcpyToSymbol(g_tile_clk_n, &d_n, sizeof d_n));
    }
    APS_CUDA(cudaMemset(d_rec, 0, nrec * 4));
    APS_CUDA(cudaMemset(d_n, 0, nw * 4));
    APS_CUDA(cudaDeviceSynchronize());
    return APS_OK;
  }
  if (!d_rec) return APS_ERR_ARGS;
  APS_CUDA(cudaDeviceSynchronize());
  APS_CUDA(cudaMemcpy(counts, d_n, nw * 4, cudaMemcpyDeviceToHost));
  APS_CUDA(cudaMemcpy(records, d_rec, nrec * 4, cudaMemcpyDeviceToHost));
  return APS_OK;
}
#endif

// Sets the shared-memory size and checks the register allocation the setmaxnreg split was computed for (a smaller one
// would leave the epilogue's setmaxnreg.inc waiting for registers that warpgroup 0 never frees).
template <typename Kern>
static int prepare_launch(Kern kern, int cs, size_t smem) {
  APS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  cudaFuncAttributes fa;
  APS_CUDA(cudaFuncGetAttributes(&fa, kern));
  if (fa.numRegs != launch_regs(cs)) {
    aps_set_error(APS_ERR_CUDA, "", "k_knn_tc allocates %d registers per thread, the register split assumes %d",
                  fa.numRegs, launch_regs(cs));
    return APS_ERR_CUDA;
  }
  return APS_OK;
}

int aps_k_knn_tc_supported(int Dp) { return Dp == 64 || Dp == 128; }
int aps_k_knn_tc_tile_rows() { return TN; }
int aps_k_knn_tc_tile_mode_stride() { return 2 * 3; }   // kcand == 3: two lists of three per row
int aps_k_knn_tc_tile_mode_segment() { return TN / 2; }  // ... each over 64-column segments of the train tiles

// Work decomposition shared by the launcher and by callers that size the candidate buffers.
struct TcSchedule {
  int units_full, tail_units, tail_seg, nslot, tiles_per_seg, tail_balanced;
  int64_t tile_lo, tile_hi;
};
static TcSchedule make_schedule(int sm_count, int64_t nq, int64_t t0, int64_t t1, bool all_segmented = false) {
  TcSchedule sc;
  sc.tail_balanced = 0;
  if (all_segmented) {
    sc.tile_lo = t0 / TN;
    sc.tile_hi = aps_ceil_div(t1, TN);
    const int64_t tiles = sc.tile_hi - sc.tile_lo;
    sc.units_full = 0;
    sc.tail_units = (int)aps_ceil_div(nq, (int64_t)RB * TM);
    sc.tail_seg = (int)(tiles < MAX_SEG ? (tiles < 1 ? 1 : tiles) : MAX_SEG);
    sc.nslot = sc.tail_seg * CSPLIT;
    sc.tiles_per_seg = (int)aps_ceil_div(tiles, sc.tail_seg);
    return sc;
  }
  sc.tile_lo = t0 / TN;
  sc.tile_hi = aps_ceil_div(t1, TN);
  const int64_t tiles = sc.tile_hi - sc.tile_lo;
  const int64_t pairs = aps_ceil_div(nq, (int64_t)RB * TM);  // 256-row query block pairs
  const int64_t grid = sm_count;  // fewer pairs than SMs: every unit is a (segmented) tail unit
  sc.units_full = (int)((pairs / grid) * grid);
  sc.tail_units = (int)(pairs - sc.units_full);
  sc.tail_seg = 1;
  if (sc.tail_units > 0) {
    // segments per tail unit: minimise the length of the last round, ceil(tail_units * s / grid) / s
    int64_t seg = 1, best_num = aps_ceil_div((int64_t)sc.tail_units, grid), best_den = 1;
    for (int64_t sg = 2; sg <= MAX_SEG && sg <= tiles; ++sg) {
      const int64_t num = aps_ceil_div((int64_t)sc.tail_units * sg, grid);
      if (num * best_den < best_num * sg) { seg = sg; best_num = num; best_den = sg; }
    }
    sc.tail_seg = (int)seg;
    // Balanced tail: cut the tail's tile steps (unit-major) into `grid` equal shares.  Length of the last round
    // = tail_units / grid exactly, at the price of up to ceil(grid / tail_units) + 1 lists per row.
    if (CSPLIT == 1 && tiles >= 8 && sc.units_full > 0) {
      const int64_t T = tiles, W = (int64_t)sc.tail_units * T, G = grid;
      int64_t max_pieces = 0;
      for (int64_t r = 0; r < sc.tail_units; ++r) {
        const int64_t own0 = ((r * T + 1) * G - 1) / W, ownl = ((r * T + T) * G - 1) / W;
        if (ownl - own0 + 1 > max_pieces) max_pieces = ownl - own0 + 1;
      }
      // worth it if it shortens the last round by more than 5 %
      if (max_pieces <= MAX_SEG && (int64_t)sc.tail_units * best_den * 100 < best_num * G * 95) {
        sc.tail_balanced = 2;
        sc.tail_seg = (int)max_pieces;
      }
      // Few tail units (cannot be cut finely enough with 4 lists): merge the last full round into the tail, so
      // that every share is >= one unit long (<= 3 pieces per CTA, <= 2 lists per row).  CTAs of that round no
      // longer sweep the tiles in lockstep, so only while the bf16 train view stays L2-resident.
      const double t_cur = sc.tail_balanced ? (double)sc.tail_units / G : (double)best_num / best_den;
      if ((double)sc.tail_units / G < 0.95 * t_cur && sc.units_full >= G && (t1 - t0) <= 393216) {
        sc.units_full -= (int)G;
        sc.tail_units += (int)G;
        sc.tail_balanced = 3;
        const int64_t W2 = (int64_t)sc.tail_units * T;
        max_pieces = 0;
        for (int64_t r = 0; r < sc.tail_units; ++r) {
          const int64_t own0 = ((r * T + 1) * G - 1) / W2, ownl = ((r * T + T) * G - 1) / W2;
          if (ownl - own0 + 1 > max_pieces) max_pieces = ownl - own0 + 1;
        }
        sc.tail_seg = (int)max_pieces;
      }
    }
  }
  sc.nslot = (sc.tail_units > 0 ? sc.tail_seg : 1) * CSPLIT;
  sc.tiles_per_seg = (int)aps_ceil_div(tiles, sc.tail_seg);
  return sc;
}
// rows [0, full_rows) of the query range belong to full-width units: their candidates are all in list 0
int64_t aps_k_knn_tc_full_rows(int sm_count, int64_t nq, int64_t t0, int64_t t1) {
  const TcSchedule sc = make_schedule(sm_count, nq, t0, t1, false);
  const int64_t rows = (int64_t)sc.units_full * RB * TM;
  return rows < nq ? rows : nq;
}
int aps_k_knn_tc_slots(int sm_count, int64_t nq, int64_t t0, int64_t t1, int all_segmented) {
  return make_schedule(sm_count, nq, t0, t1, all_segmented != 0).nslot;
}

// the raw pre-filter pays once a unit sweeps >= ~100 tiles (insert probability per chunk ~ 64 / tiles seen)
static bool use_prefilter(const TcSchedule& sc, const aps_tc_problem& p) {
  const int64_t sweep = (sc.tile_hi - sc.tile_lo) / ((sc.units_full && !p.nrows_dev) ? 1 : (sc.tail_seg > 0 ? sc.tail_seg : 1));
  return sweep >= 96 && p.tile_bounds != nullptr;
}

int aps_k_knn_tc_describe(int sm_count, const aps_tc_problem& p, int* out) {
  const TcSchedule sc = make_schedule(sm_count, p.q1 - p.q0, p.t0, p.t1, p.nrows_dev != nullptr);
  out[0] = sc.nslot;
  out[1] = use_prefilter(sc, p) ? 1 : 0;
  out[2] = sc.units_full;
  out[3] = sc.tail_units;
  out[4] = sc.tail_seg;
  out[5] = sc.tail_balanced;
  out[6] = sc.tiles_per_seg;
  return APS_OK;
}

int aps_k_knn_tc(cudaStream_t s, int sm_count, const aps_tc_problem& p, cudaEvent_t ev0, cudaEvent_t ev1) {
  if (!aps_k_knn_tc_supported(p.Dp)) {
    aps_set_error(APS_ERR_DIM, "", "tcgen05 path supports padded descriptor lengths 64 and 128 (got %d)", p.Dp);
    return APS_ERR_DIM;
  }
  if ((p.kcand != KC && p.kcand != KC_LARGE) || (p.kcand == KC_LARGE && p.dump)) {
    aps_set_error(APS_ERR_ARGS, "", "kcand must be %d or %d (score dumps: %d)", KC, KC_LARGE, KC);
    return APS_ERR_ARGS;
  }
  if (p.q1 <= p.q0 || p.t1 <= p.t0) return APS_OK;
  const TcSchedule sc = make_schedule(sm_count, p.q1 - p.q0, p.t0, p.t1, p.nrows_dev != nullptr);
  if (p.nslot != sc.nslot) {
    aps_set_error(APS_ERR_ARGS, "", "candidate buffers must be sized with aps_k_knn_tc_slots (%d != %d)", p.nslot, sc.nslot);
    return APS_ERR_ARGS;
  }
  CUtensorMap map_q, map_t;
  const CUtensorMapDataType dt = p.operand_fp16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  APS_TRY(make_map(&map_q, p.Qb, p.Fq_total, p.Dp, TM, dt));
  APS_TRY(make_map(&map_t, p.Tb, p.Ft_total, p.Dp, TN, dt));
  KParams P;
  P.q0 = p.q0; P.q1 = p.q1; P.t0 = p.t0; P.t1 = p.t1;
  P.dp = p.Dp;
  P.nslot = sc.nslot;
  P.units_full = sc.units_full;
  P.tail_units = sc.tail_units;
  P.tail_seg = sc.tail_seg;
  P.tile_lo = sc.tile_lo;
  P.tile_hi = sc.tile_hi;
  P.tiles_per_seg = sc.tiles_per_seg;
  P.tail_balanced = sc.tail_balanced;
  P.grid = sm_count;
  P.colscale = p.colscale;
  P.colbias = p.colbias;
  P.tile_bounds = p.tile_bounds;
  P.cand_idx = p.cand_idx;
  P.cand_score = p.cand_score;
  P.dump = p.dump;
  P.unit_table = nullptr;
  P.n_table_units = 0;
  P.cand_stride = p.kcand;
  P.variant_flag = nullptr;
  P.variant_want = 0;
  P.idesc = p.operand_fp16 ? make_idesc_f16_f32acc(TM, TN) : make_idesc_bf16(TM, TN);
  P.nrows_dev = p.nrows_dev;
  if (p.nrows_dev) {  // second pass: every unit in MAX_SEG column segments (more candidate lists per row)
    P.units_full = 0;
    P.tail_units = (int)aps_ceil_div(p.q1 - p.q0, (int64_t)RB * TM);
    P.tail_seg = sc.tail_seg;
    P.tiles_per_seg = sc.tiles_per_seg;
  }
  // every (row, list) slot is written by exactly one work unit (full-width units clear the unused lists)
  const size_t smem = smem_bytes(p.Dp, CSPLIT, p.kcand);
  const int64_t units = sc.tail_balanced ? (int64_t)sc.units_full + (int64_t)sc.tail_balanced * sm_count
                                         : (int64_t)sc.units_full + (int64_t)sc.tail_units * sc.tail_seg;
  const unsigned grid = (unsigned)(units < sm_count ? units : sm_count);  // upper bound in second-pass mode
  if (ev0) APS_CUDA(cudaEventRecord(ev0, s));
  auto launch = [&](auto kern) -> int {
    APS_TRY(prepare_launch(kern, CSPLIT, smem));
    kern<<<grid, NUM_THREADS, smem, s>>>(map_q, map_t, P);
    return APS_OK;
  };
  const bool pre = use_prefilter(sc, p);
  if (p.kcand == KC_LARGE) {  // 6 <= k <= 12: one launch whatever the operands (the re-rank reads all 16 slots)
    if (pre)
      APS_TRY(p.bias ? launch(k_knn_tc<true, false, true, KC_LARGE>) : launch(k_knn_tc<false, false, true, KC_LARGE>));
    else
      APS_TRY(p.bias ? launch(k_knn_tc<true, false, false, KC_LARGE>) : launch(k_knn_tc<false, false, false, KC_LARGE>));
  } else if (p.dump)
    APS_TRY(p.bias ? launch(k_knn_tc<true, true, false, KC>) : launch(k_knn_tc<false, true, false, KC>));
  else if (p.exact_flag && !p.nrows_dev) {
    // list size chosen by a device-side flag, no host round trip: both variants are launched, one exits at once
    P.variant_flag = p.exact_flag;
    P.variant_want = 1;
    if (pre)
      APS_TRY(p.bias ? launch(k_knn_tc<true, false, true, 6>) : launch(k_knn_tc<false, false, true, 6>));
    else
      APS_TRY(p.bias ? launch(k_knn_tc<true, false, false, 6>) : launch(k_knn_tc<false, false, false, 6>));
    APS_LAUNCHED();
    P.variant_want = 0;
    if (pre)
      APS_TRY(p.bias ? launch(k_knn_tc<true, false, true, KC>) : launch(k_knn_tc<false, false, true, KC>));
    else
      APS_TRY(p.bias ? launch(k_knn_tc<true, false, false, KC>) : launch(k_knn_tc<false, false, false, KC>));
  } else if (pre)
    APS_TRY(p.bias ? launch(k_knn_tc<true, false, true, KC>) : launch(k_knn_tc<false, false, true, KC>));
  else
    APS_TRY(p.bias ? launch(k_knn_tc<true, false, false, KC>) : launch(k_knn_tc<false, false, false, KC>));
  APS_LAUNCHED();
  if (ev1) APS_CUDA(cudaEventRecord(ev1, s));
  return APS_OK;
}

// gathers the bf16 operand rows listed in rows[0 .. *nrows_dev) into a compact matrix (second-pass queries)
__global__ void k_gather_rows(const uint4* __restrict__ src, const int32_t* __restrict__ rows,
                              const int32_t* __restrict__ nrows_dev, int chunks, uint4* __restrict__ dst) {
  const int64_t total = (int64_t)(*nrows_dev) * chunks;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / chunks;
    const int c = (int)(i - r * chunks);
    dst[i] = src[(int64_t)rows[r] * chunks + c];
  }
}
int aps_k_gather_rows(cudaStream_t s, const __nv_bfloat16* src, int Dp, const int32_t* rows, const int32_t* nrows_dev,
                      int64_t max_rows, __nv_bfloat16* dst) {
  if (max_rows == 0) return APS_OK;
  const int chunks = Dp * 2 / 16;
  const unsigned grid = (unsigned)aps_min64(aps_ceil_div(max_rows * chunks, 256), 148 * 8);
  k_gather_rows<<<grid, 256, 0, s>>>((const uint4*)src, rows, nrows_dev, chunks, (uint4*)dst);
  APS_LAUNCHED();
  return APS_OK;
}

// Batched launch: explicit work units, e.g. one per (256-row block of image i, image j) (pairwise) or per 256-row block
// of one image set against that set's rows (aps_feature_matching_global_sets).  One candidate list of kcand per row at
// candidate-buffer row (unit.out_row + row offset).
int aps_k_knn_tc_units(cudaStream_t s, int sm_count, const aps_tc_problem& p, const aps_tc_unit* d_units,
                       int64_t n_units) {
  if (!aps_k_knn_tc_supported(p.Dp)) {
    aps_set_error(APS_ERR_DIM, "", "tcgen05 path supports padded descriptor lengths 64 and 128 (got %d)", p.Dp);
    return APS_ERR_DIM;
  }
  if (n_units <= 0) return APS_OK;
  CUtensorMap map_q, map_t;
  const CUtensorMapDataType dt = p.operand_fp16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  APS_TRY(make_map(&map_q, p.Qb, p.Fq_total, p.Dp, TM, dt));
  APS_TRY(make_map(&map_t, p.Tb, p.Ft_total, p.Dp, TN, dt));
  KParams P;
  memset(&P, 0, sizeof P);
  P.idesc = p.operand_fp16 ? make_idesc_f16_f32acc(TM, TN) : make_idesc_bf16(TM, TN);
  P.nrows_dev = nullptr;
  P.dp = p.Dp;
  P.nslot = 1;
  P.colscale = p.colscale;
  P.colbias = p.colbias;
  P.tile_bounds = p.tile_bounds;
  P.cand_idx = p.cand_idx;
  P.cand_score = p.cand_score;
  P.dump = nullptr;
  P.unit_table = d_units;
  P.n_table_units = n_units;
  P.cand_stride = p.kcand;
  const int cs_groups = p.kcand == 3 ? 2 : CSPLIT;  // epilogue groups per row block of the variant launched below
  const size_t smem = smem_bytes(p.Dp, cs_groups, p.kcand == KC_LARGE ? KC_LARGE : KC);
  const unsigned grid = (unsigned)(n_units < sm_count ? n_units : sm_count);
  const int threads = threads_for(cs_groups);
  auto launch = [&](auto kern) -> int {
    APS_TRY(prepare_launch(kern, cs_groups, smem));
    kern<<<grid, threads, smem, s>>>(map_q, map_t, P);
    return APS_OK;
  };
  if (p.kcand == 3) {  // short sweeps: branch-free two-best per segment, two epilogue groups (lists) per row block
    P.cand_stride = aps_k_knn_tc_tile_mode_stride();
    APS_TRY(p.bias ? launch(k_knn_tc<true, false, false, 3, 2>) : launch(k_knn_tc<false, false, false, 3, 2>));
  } else if (p.kcand == 4)
    APS_TRY(p.bias ? launch(k_knn_tc<true, false, false, 4>) : launch(k_knn_tc<false, false, false, 4>));
  else if (p.kcand == KC)
    APS_TRY(p.bias ? launch(k_knn_tc<true, false, false, KC>) : launch(k_knn_tc<false, false, false, KC>));
  else if (p.kcand == KC_LARGE)  // the K' = 16 lists of 6 <= k <= 12 (batched global sets)
    APS_TRY(p.bias ? launch(k_knn_tc<true, false, false, KC_LARGE>) : launch(k_knn_tc<false, false, false, KC_LARGE>));
  else {
    aps_set_error(APS_ERR_ARGS, "", "kcand must be 3, 4, %d or %d", KC, KC_LARGE);
    return APS_ERR_ARGS;
  }
  APS_LAUNCHED();
  return APS_OK;
}
