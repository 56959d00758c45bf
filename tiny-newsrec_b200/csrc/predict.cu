// Prediction files for unlabeled impressions: the rank of every candidate within its impression under the eval scores,
// and the MIND prediction text ("<impression id> [r_1,r_2,...,r_C]\n" per impression) built on the device.
//
//   predict_rank_kernel   warp per impression.  The order keys of its scores sit in shared memory; lane l ranks
//                         candidates l, l + 32, ... (PR_OWN per pass over the keys, all in registers) as
//                         rank_c = 1 + #{s_j > s_c} + #{s_j == s_c, j > c}, the rank eval_rank_kernel gives a positive
//                         (np.argsort(score, kind="stable")[::-1] order; -0 == +0).  Every key read is a broadcast.
//                         MIND impressions hold 2 to 300 candidates (mean ~37): O(C^2 / 32) compares per warp.
//   predict_line_bytes_kernel / predict_write_kernel
//                         warp per impression: the byte length of every line (scanned by CUB into line offsets), then
//                         the text itself -- lanes turn their ranks into digits and a warp prefix sum of the lengths
//                         places them after "<id> [".
#include "common.cuh"
#include "eval_score.cuh"
#include <cub/device/device_scan.cuh>

#define TNR_API extern "C" __attribute__((visibility("default")))

namespace tnr {

constexpr int PR_WARPS = 4;
constexpr int PR_OWN = 2;            // candidates a lane ranks per pass over the keys (one pass covers C <= 64)
constexpr int PR_MAX_C = 51200;      // 200 KB of keys for one warp

__global__ void __launch_bounds__(PR_WARPS * 32)
predict_rank_kernel(const float* __restrict__ score, const long long* __restrict__ ptr, long long n_imp, int cap,
                    int32_t* __restrict__ rank) {
  extern __shared__ __align__(16) uint32_t s_key_all[];
  const int warp = uniform_warp_id(), lane = threadIdx.x & 31;
  const long long b = (long long)blockIdx.x * (blockDim.x >> 5) + warp;
  if (b >= n_imp) return;
  uint32_t* s_key = s_key_all + (size_t)warp * cap;
  const long long p0 = ptr[b];
  const int C = (int)(ptr[b + 1] - p0);
  const int C4 = (C + 3) & ~3;       // whole 4-key groups: key 0 (no finite float maps to it) ranks below every score
  for (int c = lane; c < C4; c += 32) s_key[c] = c < C ? order_key(score[p0 + c]) : 0u;
  __syncwarp();
  for (int c0 = 0; c0 < C; c0 += 32 * PR_OWN) {
    uint32_t kc[PR_OWN];
    int above[PR_OWN];
#pragma unroll
    for (int r = 0; r < PR_OWN; ++r) {
      const int c = c0 + 32 * r + lane;
      kc[r] = c < C ? s_key[c] : 0xffffffffu;
      above[r] = 0;
    }
    for (int g = 0; g < C4; g += 4) {
      const uint4 k4 = *reinterpret_cast<const uint4*>(s_key + g);
      const uint32_t kj[4] = {k4.x, k4.y, k4.z, k4.w};
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int r = 0; r < PR_OWN; ++r)
          above[r] += (int)(kj[u] > kc[r]) | ((int)(kj[u] == kc[r]) & (int)(g + u > c0 + 32 * r + lane));
    }
#pragma unroll
    for (int r = 0; r < PR_OWN; ++r) {
      const int c = c0 + 32 * r + lane;
      if (c < C) rank[p0 + c] = above[r] + 1;
    }
  }
}

__device__ __forceinline__ int dec_digits(unsigned long long v) {     // decimal digits of v (0 has one)
  int n = 1;
  unsigned long long p = 10ull;
#pragma unroll 1
  for (; n < 20 && v >= p; ++n) p *= 10ull;
  return n;
}

__device__ __forceinline__ int rank_chars(int v) {                    // length of the decimal text of an int32
  const unsigned u = v < 0 ? 0u - (unsigned)v : (unsigned)v;
  return (v < 0) + dec_digits(u);
}

__device__ __forceinline__ unsigned long long pow10u(int e) {
  unsigned long long p = 1ull;
#pragma unroll 1
  for (int i = 0; i < e; ++i) p *= 10ull;
  return p;
}

constexpr int PF_WARPS = 8;

// bytes[b] = the length of line b ("<id> [" + ranks joined by ',' + "]\n"); bytes[n_imp] = 0 (the scan's total)
__global__ void __launch_bounds__(PF_WARPS * 32)
predict_line_bytes_kernel(const long long* __restrict__ imp_id, const long long* __restrict__ ptr,
                          const int32_t* __restrict__ rank, long long n_imp, long long* __restrict__ bytes) {
  const int lane = threadIdx.x & 31;
  const long long b = (long long)blockIdx.x * PF_WARPS + uniform_warp_id();
  if (b > n_imp) return;
  if (b == n_imp) {
    if (lane == 0) bytes[b] = 0;
    return;
  }
  const long long p0 = ptr[b];
  const int C = (int)(ptr[b + 1] - p0);
  int n = 0;
  for (int c = lane; c < C; c += 32) n += rank_chars(rank[p0 + c]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) n += __shfl_xor_sync(0xffffffffu, n, o);
  if (lane == 0) bytes[b] = (long long)dec_digits((unsigned long long)imp_id[b]) + 2 + n + (C > 0 ? C - 1 : 0) + 2;
}

__global__ void __launch_bounds__(PF_WARPS * 32)
predict_write_kernel(const long long* __restrict__ imp_id, const long long* __restrict__ ptr,
                     const int32_t* __restrict__ rank, long long n_imp, const long long* __restrict__ line_off,
                     uint8_t* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const long long b = (long long)blockIdx.x * PF_WARPS + uniform_warp_id();
  if (b >= n_imp) return;
  const long long p0 = ptr[b];
  const int C = (int)(ptr[b + 1] - p0);
  long long o = line_off[b];
  const unsigned long long id = (unsigned long long)imp_id[b];
  const int il = dec_digits(id);
  if (lane < il) out[o + il - 1 - lane] = (uint8_t)('0' + (id / pow10u(lane)) % 10ull);     // lane l: digit l from the right
  if (lane == 0) {
    out[o + il] = ' ';
    out[o + il + 1] = '[';
  }
  o += il + 2;
  for (int c0 = 0; c0 < C; c0 += 32) {
    const int c = c0 + lane;
    const int v = c < C ? rank[p0 + c] : 0;
    const int len = c < C ? rank_chars(v) + (c < C - 1) : 0;           // the text and its comma
    int incl = len;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= d) incl += t;
    }
    if (c < C) {
      long long q = o + incl - len;
      unsigned u = (unsigned)v;
      if (v < 0) {
        out[q++] = '-';
        u = 0u - u;
      }
      const int nd = dec_digits(u);
      for (int k = nd - 1; k >= 0; --k) {
        out[q + k] = (uint8_t)('0' + u % 10u);
        u /= 10u;
      }
      if (c < C - 1) out[q + nd] = ',';
    }
    o += __shfl_sync(0xffffffffu, incl, 31);
  }
  if (lane == 0) {
    out[o] = ']';
    out[o + 1] = '\n';
  }
}

static int pf_scan_bytes(long long n_imp, size_t& bytes) {
  bytes = 0;
  return cub::DeviceScan::ExclusiveSum(nullptr, bytes, (long long*)nullptr, n_imp + 1) != cudaSuccess;
}

}  // namespace tnr

using namespace tnr;

TNR_API int tnr_predict_ranks(const float* table, long long n_rows, const float* user, const long long* ptr,
                              const int32_t* cand, long long n_imp, long long nnz, int D, int max_c, float* scores,
                              int32_t* ranks, void* stream) {
  TNR_REQUIRE(D % 32 == 0 && D >= 32 && D <= 512, "tnr_predict_ranks: D=%d must be a multiple of 32 in 32..512", D);
  TNR_REQUIRE(n_rows >= 1, "tnr_predict_ranks: empty table");
  TNR_REQUIRE(max_c >= 0 && max_c <= PR_MAX_C, "tnr_predict_ranks: max candidates %d outside 0..%d", max_c, PR_MAX_C);
  TNR_REQUIRE(nnz == 0 || (scores != nullptr && ranks != nullptr), "tnr_predict_ranks: scores and ranks are required");
  if (n_imp == 0 || nnz == 0) return 0;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (eval_scores("tnr_predict_ranks", table, n_rows, user, ptr, cand, n_imp, nnz, D, scores, st)) return 1;
  const int cap = ((max_c > 1 ? max_c : 1) + 3) & ~3;
  int wpb = PR_WARPS;
  while (wpb > 1 && (size_t)wpb * cap * 4 > 160 * 1024) wpb >>= 1;
  const size_t smem = (size_t)wpb * cap * 4;
  if (smem > 48 * 1024) TNR_SET_SMEM(predict_rank_kernel, smem);
  predict_rank_kernel<<<(unsigned)((n_imp + wpb - 1) / wpb), wpb * 32, smem, st>>>(scores, ptr, n_imp, cap, ranks);
  TNR_LAUNCH_CHECK();
  return 0;
}

TNR_API long long tnr_predict_format_ws_bytes(long long n_imp) {
  if (n_imp < 0) return -1;
  size_t bytes = 0;
  if (pf_scan_bytes(n_imp, bytes)) return -1;
  return (long long)bytes;
}

TNR_API int tnr_predict_format_size(const long long* imp_id, const long long* ptr, const int32_t* ranks, long long n_imp,
                                    long long* line_off, void* workspace, long long ws_bytes, void* stream) {
  TNR_REQUIRE(n_imp >= 0 && line_off != nullptr, "tnr_predict_format_size: line_off int64 [n_imp + 1] is required");
  size_t need = 0;
  TNR_REQUIRE(pf_scan_bytes(n_imp, need) == 0, "tnr_predict_format_size: scan size query failed");
  TNR_REQUIRE(ws_bytes >= (long long)need && (need == 0 || workspace != nullptr),
              "tnr_predict_format_size: workspace of %lld bytes needed (tnr_predict_format_ws_bytes), got %lld",
              (long long)need, ws_bytes);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  predict_line_bytes_kernel<<<(unsigned)((n_imp + 1 + PF_WARPS - 1) / PF_WARPS), PF_WARPS * 32, 0, st>>>(
      imp_id, ptr, ranks, n_imp, line_off);
  TNR_LAUNCH_CHECK();
  TNR_CHECK_CUDA(cub::DeviceScan::ExclusiveSum(workspace, need, line_off, n_imp + 1, st));
  return 0;
}

TNR_API int tnr_predict_format_write(const long long* imp_id, const long long* ptr, const int32_t* ranks, long long n_imp,
                                     const long long* line_off, uint8_t* out, void* stream) {
  TNR_REQUIRE(n_imp >= 0 && line_off != nullptr && (n_imp == 0 || out != nullptr),
              "tnr_predict_format_write: line_off and out are required");
  if (n_imp == 0) return 0;
  predict_write_kernel<<<(unsigned)((n_imp + PF_WARPS - 1) / PF_WARPS), PF_WARPS * 32, 0,
                         reinterpret_cast<cudaStream_t>(stream)>>>(imp_id, ptr, ranks, n_imp, line_off, out);
  TNR_LAUNCH_CHECK();
  return 0;
}
