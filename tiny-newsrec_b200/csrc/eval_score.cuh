// The eval score of one (news row, user) pair and the order it ranks by, shared by the impression scoring kernels
// (misc_kernels.cu) and the top-k recommendation kernels (recommend.cu): a recommended news carries bit for bit the
// score tnr_eval_metrics gives it as a candidate.
#pragma once
#include "common.cuh"

namespace tnr {

// One row's fp32 dot product over an 8-lane group (D = 32 * VPL): lane gl of the group holds float4 gl + 8 v of the row
// (x) and of the user vector (u).  Every lane of the group returns the same sum, and the summation tree is the same for
// every row and user, so duplicate rows tie exactly.  All 32 lanes of the warp must call it (the groups meet in
// shuffles).
template <int VPL>
__device__ __forceinline__ float eval_dot8(const float4 (&x)[VPL], const float4 (&u)[VPL]) {
  float t = 0.f;
#pragma unroll
  for (int v = 0; v < VPL; ++v)
    t = fmaf(x[v].x, u[v].x, fmaf(x[v].y, u[v].y, fmaf(x[v].z, u[v].z, fmaf(x[v].w, u[v].w, t))));
  t += __shfl_xor_sync(0xffffffffu, t, 1);
  t += __shfl_xor_sync(0xffffffffu, t, 2);
  t += __shfl_xor_sync(0xffffffffu, t, 4);
  return t;
}

__device__ __forceinline__ uint32_t order_key(float f) {     // a < b  <=>  key(a) < key(b)   (-0 == +0 kept equal)
  const uint32_t u = __float_as_uint(f + 0.0f);               // -0.0f + 0.0f = +0.0f
  return u ^ ((uint32_t)((int32_t)u >> 31) | 0x80000000u);
}

// Host: launches the flat scoring kernel of tnr_eval_metrics (misc_kernels.cu) on `st`: scores fp32 [nnz] of a CSR
// batch (ptr int64 [n_imp + 1], cand int32 [nnz]), D in {32, 64, 128, 256, 512}.  Returns 0, or 1 with the error set
// (prefixed by `what`).
int eval_scores(const char* what, const float* table, long long n_rows, const float* user, const long long* ptr,
                const int32_t* cand, long long n_imp, long long nnz, int D, float* scores, cudaStream_t st);

}  // namespace tnr
