// aps_exact_math.cuh -- the oracle's float operation orders as device functions (explicit _rn
// intrinsics: no FMA contraction), shared by the re-rank and the pairwise fallback kernels.
#pragma once
#include <math_constants.h>

#include "aps_common.cuh"

__device__ __forceinline__ float l2sq_flann(const float* __restrict__ a, const float* __restrict__ b, int D) {
  float result = 0.f;
  int d = 0;
  for (; d + 3 < D; d += 4) {
    float4 x, y;
    if ((D & 3) == 0) {
      x = *reinterpret_cast<const float4*>(a + d);
      y = *reinterpret_cast<const float4*>(b + d);
    } else {
      x = make_float4(a[d], a[d + 1], a[d + 2], a[d + 3]);
      y = make_float4(b[d], b[d + 1], b[d + 2], b[d + 3]);
    }
    float e0 = __fsub_rn(x.x, y.x), e1 = __fsub_rn(x.y, y.y), e2 = __fsub_rn(x.z, y.z), e3 = __fsub_rn(x.w, y.w);
    float s = __fadd_rn(__fmul_rn(e0, e0), __fmul_rn(e1, e1));
    s = __fadd_rn(s, __fmul_rn(e2, e2));
    s = __fadd_rn(s, __fmul_rn(e3, e3));
    result = __fadd_rn(result, s);
  }
  for (; d < D; ++d) {
    float e0 = __fsub_rn(a[d], b[d]);
    result = __fadd_rn(result, __fmul_rn(e0, e0));
  }
  return result;
}

// The sequential helpers below read both rows with 128-bit loads when the rows allow it (length a multiple of four,
// 16-byte aligned -- every row of a cudaMalloc'ed [rows x D] matrix then): a lane that owns a train row otherwise
// issues four times the load instructions and touches each 32-byte sector eight times.  The ORDER of the float
// operations is the scalar loop's: same bits.
__device__ __forceinline__ bool rows_vec4(const float* a, const float* b, int D) {
  return ((D & 3) == 0) && ((((uintptr_t)a | (uintptr_t)b) & 15u) == 0);
}
__device__ __forceinline__ float dot_seq(const float* __restrict__ a, const float* __restrict__ b, int D);
__device__ __forceinline__ float ssd_seq(const float* __restrict__ a, const float* __restrict__ b, int D, float a2,
                                         float b2) {
  const float g = dot_seq(a, b, D);
  return __fsub_rn(__fadd_rn(a2, b2), __fmul_rn(2.0f, g));
}

// metric 2: plain squared Euclidean distance, sequential over the columns (the 'kdtree' / 'subsetpdist2' branches of
// matchFeaturesScratch.m:142-155 search by EUCLIDEAN distance -- knnsearch / pdist2 -- and square it afterwards):
// the caller ranks by sqrt_rn(s) and reports fmul_rn(r, r).
__device__ __forceinline__ float l2sq_seq(const float* __restrict__ a, const float* __restrict__ b, int D) {
  float s = 0.f;
  if (rows_vec4(a, b, D)) {
    for (int d = 0; d < D; d += 4) {
      const float4 x = *reinterpret_cast<const float4*>(a + d), y = *reinterpret_cast<const float4*>(b + d);
      float e = __fsub_rn(x.x, y.x);
      s = __fadd_rn(s, __fmul_rn(e, e));
      e = __fsub_rn(x.y, y.y);
      s = __fadd_rn(s, __fmul_rn(e, e));
      e = __fsub_rn(x.z, y.z);
      s = __fadd_rn(s, __fmul_rn(e, e));
      e = __fsub_rn(x.w, y.w);
      s = __fadd_rn(s, __fmul_rn(e, e));
    }
    return s;
  }
  for (int d = 0; d < D; ++d) {
    const float e = __fsub_rn(a[d], b[d]);
    s = __fadd_rn(s, __fmul_rn(e, e));
  }
  return s;
}

// metric 3 ('pca2nn', matchFeaturesScratch.m:536-573 doBlock): cosine similarity of the projected, normalised rows,
// G = A*B.' restated as a sequential float32 dot; the caller ranks by -sim and reports fl(2 - fl(2 sim)).
__device__ __forceinline__ float dot_seq(const float* __restrict__ a, const float* __restrict__ b, int D) {
  float g = 0.f;
  if (rows_vec4(a, b, D)) {
    for (int d = 0; d < D; d += 4) {
      const float4 x = *reinterpret_cast<const float4*>(a + d), y = *reinterpret_cast<const float4*>(b + d);
      g = __fadd_rn(g, __fmul_rn(x.x, y.x));
      g = __fadd_rn(g, __fmul_rn(x.y, y.y));
      g = __fadd_rn(g, __fmul_rn(x.z, y.z));
      g = __fadd_rn(g, __fmul_rn(x.w, y.w));
    }
    return g;
  }
  for (int d = 0; d < D; ++d) g = __fadd_rn(g, __fmul_rn(a[d], b[d]));
  return g;
}

// error bound of the approximate distance; flags: [0] operands exact in bf16, [1] bits of max|sq-1|,
// [2] bits of max sq.  See DESIGN.md "Exactness of the tensor-core search".
// operand_kind: 0 bf16 (flags[0] = rows exact in bf16), 1 fp16 never exact, 2 fp16 (flags[0] = rows exact in fp16)
__device__ __forceinline__ float eps_bound(const int32_t* __restrict__ flags, int bias_mode, int operand_kind = 0) {
  const bool operand_fp16 = operand_kind != 0;
  const bool exact = flags[0] != 0 && operand_kind != 1;
  const float dev = __int_as_float(flags[1]);
  const float maxsq = fmaxf(__int_as_float(flags[2]), 1.0f);
  const float slop = 1.0e-4f * maxsq;                     // fp32 evaluation-order differences
  // operand rounding, unit roundoff u (bf16 2^-8, fp16 2^-11): |a.b - a~.b~| <= (2u + u^2) |a||b|, twice that in the
  // distance: bf16 2 * 2^-7 * (1+2^-9) * |a||b| ; fp16 2 * 2^-10 * (1+2^-12) * |a||b| (values below the fp16 normal range
  // lose at most 2^-25 each: inside `slop` for |x| <= 2).  tests/test_gpu_tc_contract.py plants rows that reach 0.85 of it.
  const float bf = exact ? 0.0f : (operand_fp16 ? 2.0e-3f : 1.57e-2f) * maxsq;
  return bias_mode ? (slop + bf) : (slop + bf + dev);     // normalised rows: |sq_b - 1| <= dev is ignored by the score
}

