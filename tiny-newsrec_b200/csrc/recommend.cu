// Top-k news recommendation over the whole news table, exact under the eval scores (eval_score.cuh).
//
// For user b the score of table row j is s(b, j) = eval_dot8(table[j], user[b]): bit for bit the score tnr_eval_metrics
// gives row j as a candidate of an impression with user vector user[b].  The table scored may be a candidate pool
// (tnr_recommend_pool): rows 1..P copied from the news table in ascending id order, local row 0 a sentinel, and `map`
// giving each local row's table id.  A copied row scores bit for bit as the original, and ascending ids keep the
// (row asc) tie order, so the kernels work in local rows and map them when they write the result.  The eligible rows
// of user b are the rows 1..n_rows-1, minus the excluded rows -- the live history with exclude_history (mask != 0,
// id != 0) and the user's exclusion list, both as local rows (ids outside the table or the pool are dropped) -- and,
// with categories, only rows whose category bit is set in the user's 64-bit mask.  The result is the top k eligible
// rows by (score desc, row asc), -1 / -inf past the last eligible row.  The B x n_rows score matrix is never written:
//
//   stage 1  rec_select_kernel: candidate selection on the tensor cores.  TF32 scores t(b, j) of a 256-user pair tile
//            against 256-row table tiles (tcgen05.mma.cta_group::2.kind::tf32, M = 256 users per CTA pair, N = 256 rows,
//            K = D).  The users of a pair stay resident in shared memory (128 KB per CTA at D = 256); table rows stream
//            through a TMA ring.  A thread of the epilogue owns a user (a TMEM lane).  The grid is split over (user tile,
//            table slice), slice-major, so the pairs running at the same time read the same slices: the table comes from
//            HBM about once per wave and from L2 for the other user tiles.  Per (user, slice) a list in global memory
//            keeps every row of an allowed category with t >= theta - 2 eps_b (the category is checked at append time,
//            only for rows that pass the threshold).  theta starts at -inf and is raised when the list fills: the
//            epilogue warp compacts the list, dropping row 0 and the excluded rows (binary search over the user's
//            sorted exclusion list; never on the per-element path) and then the rows below (the k-th best remaining
//            t) - 2 eps_b (bisection over the order keys, entries in registers).  A list that cannot be compacted below
//            its capacity has overflowed.
//            Invariant: the list holds every eligible row of the slice seen so far with t >= theta - 2 eps_b, and theta
//            is the k-th best t of eligible rows in the list (-inf while there are fewer than k), so theta never exceeds
//            the slice's k-th best eligible t.
//   stage 2  rec_merge_kernel, a block per user: the union of the user's slice lists, minus row 0 and the excluded rows
//            (a list compacted last before the end of its slice may still hold them); theta* = the union's k-th best t;
//            the rows with t >= theta* - 2 eps_b are re-scored with eval_dot8 and the exact top k taken by (score desc,
//            row asc).  Every row of the exact top k has t >= theta* - 2 eps_b (below), each slice's theta is <= theta*
//            (the union holds that slice's k eligible rows with t >= theta), so every such row is in its slice's list
//            and this is exact.
//   fallback rec_exact_kernel: a user with an overflowed list (many rows within 2 eps of theta, e.g. duplicated rows, or
//            a zero user vector) or a union too large for stage 2 is scored against every eligible row with eval_dot8,
//            under the same three filters.
//
// Exactness.  eps_b bounds |t(b, j) - s(b, j)| for every row j.  With x = table[j], u = user[b], |.| the 2-norm:
//   - tcgen05 kind::tf32 reads the fp32 operands truncated to a 10-bit mantissa: x~ = x (1 - a), |a| < 2^-10, same for u,
//     so |sum x~ u~ - sum x u| <= (2^-9 + 2^-20) sum |x_i u_i| <= (2^-9 + 2^-20) |x| |u|  (Cauchy-Schwarz);
//   - the tensor core's fp32 accumulation of D products, in any order and with truncating or rounding adds (unit error
//     2^-23): <= 1.01 D 2^-23 (1 + 2^-9) |x| |u|;
//   - the eval kernel's fp32 sum (fma chains of D / 8, three adds, round to nearest): <= 1.01 D 2^-24 |x| |u|.
//   Together < (2^-9 + 0.4 D 2^-21) |x| |u| for D >= 32.  We take eps_b = (2^-8 + D 2^-20) |u_b| R + 2^-100, R the
//   largest row norm of the table scored (of the pool, when there is one): twice that, which also covers the fp32
//   evaluation of the two norms and of theta - 2 eps (relative errors ~ D 2^-24), and an absolute term for flushed
//   subnormal products.  A loose bound only costs candidates.
//   If theta* is the k-th best eligible t, the k rows that reach it have s >= theta* - eps, so the k-th best eligible
//   s is >= theta* - eps, and a row of the exact top k has t >= s - eps >= theta* - 2 eps.
// Finite inputs are assumed.
#include <cuda.h>
#include "common.cuh"
#include "eval_score.cuh"
#include "tc_ptx.cuh"

#define TNR_API extern "C" __attribute__((visibility("default")))

namespace tnr {
namespace {

constexpr int RS_ROWS = 128;                 // users per CTA (TMEM lanes); 256 per pair
constexpr int RS_TN = 256;                   // table rows per tile (UMMA N); 128 staged by each CTA of the pair
constexpr int RS_KB = 32;                    // floats per k-block: one 128-byte swizzle row
constexpr int RS_BOX_BYTES = 128 * 128;      // one k-block of 128 rows (users or table rows): 16 KB
constexpr int RS_STAGES = 5;                 // table ring depth
constexpr int RS_DMAX = 256;
constexpr int RS_THREADS = 192;              // epilogue warps 0-3, MMA warp 4, TMA / TMEM warp 5
constexpr int RS_NBARS = 2 * RS_STAGES + 6;
constexpr int RS_CAP = 512;                  // entries of one (user, slice) candidate list
constexpr int RS_MAX_SLICES = 16;
constexpr int RM_THREADS = 256;
constexpr int RM_UCAP = 8192;                // union entries stage 2 takes; more -> the exact pass
constexpr int RX_CHUNK = 2048;               // rows per round of the exact pass
constexpr int RS_MAX_EXCL = 1024;            // excluded rows per user: H <= 512 history + E <= 512 listed
constexpr int RP_ROWS = 1024;                // rows per block of the pool compaction (4 per thread)

__host__ __device__ constexpr int rs_smem_bytes(int D) {
  return (D / RS_KB) * RS_BOX_BYTES + RS_STAGES * RS_BOX_BYTES + RS_NBARS * 8 + 16 + 1024 /*align slack*/;
}

struct RecWs {                 // views of the caller's workspace (rec_layout)
  float* hdr;                  // [0] largest table row norm (as float bits, atomicMax), [1] exact-pass user count (int)
  float* eps2;                 // [B] 2 eps_b
  int* excl;                   // [B, P] excluded local rows, ascending, INT_MAX padded (P = 0 without exclusion)
  int* cnt;                    // [S, B] list lengths; > RS_CAP: overflowed
  int* fb;                     // [B] users for the exact pass
  int2* lists;                 // [S, B, RS_CAP] (t bits, row)
};

struct RecShape {
  int S, tiles_per_slice, n_tiles, n_utiles, P;
};

static int pow2_at_least(int h) {
  int p = 1;
  while (p < h) p <<= 1;
  return p;
}

// Slices of the table: the count that minimises the pair's critical path (waves of (user tile, slice) items x tiles per
// slice), the smallest on ties (fewer lists to merge).
static RecShape rec_shape(long long n_rows, int B, int H, int exclude, int E) {
  RecShape s;
  s.n_tiles = (int)((n_rows + RS_TN - 1) / RS_TN);
  s.n_utiles = (B + 2 * RS_ROWS - 1) / (2 * RS_ROWS);
  const int pairs = num_sms() / 2;
  long long best = -1;
  int best_s = 1;
  for (int S = 1; S <= RS_MAX_SLICES && S <= s.n_tiles; ++S) {
    const int tps = (s.n_tiles + S - 1) / S;
    const int S_eff = (s.n_tiles + tps - 1) / tps;
    const long long waves = ((long long)s.n_utiles * S_eff + pairs - 1) / pairs;
    const long long cost = waves * tps;
    if (best < 0 || cost < best) { best = cost; best_s = S; }
  }
  s.tiles_per_slice = (s.n_tiles + best_s - 1) / best_s;
  s.S = (s.n_tiles + s.tiles_per_slice - 1) / s.tiles_per_slice;
  const int n_ex = (exclude ? H : 0) + E;
  s.P = n_ex > 0 ? pow2_at_least(n_ex) : 0;
  return s;
}

static size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

static size_t rec_layout(const RecShape& s, int B, char* base, RecWs* w) {
  size_t off = 0;
  auto take = [&](size_t bytes) { char* p = base ? base + off : nullptr; off += align256(bytes); return p; };
  char* hdr = take(16);
  char* eps2 = take((size_t)B * 4);
  char* excl = take((size_t)B * s.P * 4);
  char* cnt = take((size_t)s.S * B * 4);
  char* fb = take((size_t)B * 4);
  char* lists = take((size_t)s.S * B * RS_CAP * 8);
  if (w) {
    w->hdr = reinterpret_cast<float*>(hdr); w->eps2 = reinterpret_cast<float*>(eps2);
    w->excl = reinterpret_cast<int*>(excl); w->cnt = reinterpret_cast<int*>(cnt); w->fb = reinterpret_cast<int*>(fb);
    w->lists = reinterpret_cast<int2*>(lists);
  }
  return off;
}

__device__ __forceinline__ float key_to_float(uint32_t k) {     // inverse of order_key (+0 for -0)
  return __uint_as_float((k & 0x80000000u) ? (k ^ 0x80000000u) : ~k);
}
// (score desc, row asc) as one unsigned order; 0 is below every real key (order_key(-inf) > 0)
__device__ __forceinline__ uint64_t rank_key(float s, int row) {
  return ((uint64_t)order_key(s) << 32) | (uint64_t)(0xffffffffu - (uint32_t)row);
}

// ------------------------------------------------------------------------------------------------ norms and exclusions
// hdr[0] = max_j |table[j]| (fp32; non-negative floats order as their bits)
__global__ void __launch_bounds__(256) rec_table_norm_kernel(const float* __restrict__ table, long long n_rows, int D,
                                                             float* __restrict__ hdr) {
  const int lane = threadIdx.x & 31;
  float mx = 0.f;
  for (long long r = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < n_rows;
       r += ((long long)gridDim.x * blockDim.x) >> 5) {
    float s = 0.f;
    for (int d = lane; d < D; d += 32) { const float v = table[r * D + d]; s = fmaf(v, v, s); }
    mx = fmaxf(mx, sqrtf(warp_sum(s)));
  }
  mx = warp_max(mx);
  if (lane == 0) atomicMax(reinterpret_cast<unsigned*>(hdr), __float_as_uint(mx));
}

// Table id -> local row of the table scored: the id itself without a pool, else its index in the ascending pool ids
// (binary search); INT_MAX when the row is not there.
__device__ __forceinline__ int local_row(const int32_t* __restrict__ pool, long long n_rows, int id) {
  if (pool == nullptr) return id < n_rows ? id : INT_MAX;
  int lo = 0;
  for (int step = 1 << (31 - __clz((int)n_rows)); step > 0; step >>= 1)
    if (lo + step < n_rows && pool[lo + step] <= id) lo += step;
  return pool[lo] == id ? lo : INT_MAX;
}

// Block per user: 2 eps_b and the sorted exclusion list: the live history (H = 0 without exclude_history) and the
// user's E listed ids, as local rows, INT_MAX padded to P (bitonic sort of P <= 1024 ids).  Ids <= 0 and ids outside
// the table or the pool are dropped (row 0 is never eligible anyway).
__global__ void __launch_bounds__(256) rec_prep_kernel(const float* __restrict__ user, int D, const int32_t* __restrict__ hidx,
                                                       const float* __restrict__ hmask, int H, const int32_t* __restrict__ xidx,
                                                       int E, const int32_t* __restrict__ pool, long long n_rows, RecWs w,
                                                       int P) {
  __shared__ int s_id[RS_MAX_EXCL];
  __shared__ float s_red[8];
  const int b = blockIdx.x, t = threadIdx.x, lane = t & 31, warp = t >> 5;
  float sq = 0.f;
  for (int d = t; d < D; d += 256) { const float v = user[(size_t)b * D + d]; sq = fmaf(v, v, sq); }
  for (int i = t; i < P; i += 256) {
    int id = 0;
    if (i < H) id = hmask[(size_t)b * H + i] != 0.f ? hidx[(size_t)b * H + i] : 0;
    else if (i < H + E) id = xidx[(size_t)b * E + (i - H)];
    s_id[i] = id > 0 ? local_row(pool, n_rows, id) : INT_MAX;
  }
  sq = warp_sum(sq);
  if (lane == 0) s_red[warp] = sq;
  __syncthreads();
  if (t == 0) {
    float q = 0.f;
    for (int i = 0; i < 8; ++i) q += s_red[i];
    const float R = __uint_as_float(reinterpret_cast<const unsigned*>(w.hdr)[0]);
    const float eps = (0.00390625f + (float)D * 9.5367431640625e-07f) * sqrtf(q) * R + 7.888609052210118e-31f;
    w.eps2[b] = 2.0f * eps;
  }
  for (int len = 2; len <= P; len <<= 1)
    for (int j = len >> 1; j > 0; j >>= 1) {
      __syncthreads();
      for (int i = t; i < P; i += 256) {
        const int p = i ^ j;
        if (p > i) {
          const int a = s_id[i], c = s_id[p];
          const bool up = (i & len) == 0;
          if ((a > c) == up) { s_id[i] = c; s_id[p] = a; }
        }
      }
    }
  __syncthreads();
  for (int i = t; i < P; i += 256) w.excl[(size_t)b * P + i] = s_id[i];
}

// ------------------------------------------------------------------------------------------------ candidate pool
// Stream compaction of the pool mask (rows >= 1 with mask != 0), in three passes: per-block counts, one block's
// exclusive scan of the counts, and the ordered write.  ids[0] = 0 is the sentinel row; ids[1..P] ascending.

// Exclusive block scan of v (blockDim.x a multiple of 32); *total = the block's sum.  sh: 33 ints.
__device__ __forceinline__ int block_scan_excl(int v, int* sh, int* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  int inc = v;
  for (int o = 1; o < 32; o <<= 1) {
    const int u = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += u;
  }
  if (lane == 31) sh[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    int x = lane < nw ? sh[lane] : 0;
    for (int o = 1; o < 32; o <<= 1) {
      const int u = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += u;
    }
    if (lane < nw) sh[lane] = x;
    if (lane == 31) sh[32] = x;
  }
  __syncthreads();
  const int r = (warp > 0 ? sh[warp - 1] : 0) + inc - v;
  *total = sh[32];
  __syncthreads();
  return r;
}

__device__ __forceinline__ int pool_flags(const uint8_t* __restrict__ mask, long long n_rows, long long r0) {
  int f = 0;
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const long long r = r0 + q;
    if (r >= 1 && r < n_rows && mask[r] != 0) f |= 1 << q;
  }
  return f;
}

__global__ void __launch_bounds__(256) rec_pool_count_kernel(const uint8_t* __restrict__ mask, long long n_rows,
                                                             int* __restrict__ cnt) {
  __shared__ int sh[33];
  const int f = pool_flags(mask, n_rows, (long long)blockIdx.x * RP_ROWS + 4 * threadIdx.x);
  int total;
  block_scan_excl(__popc(f), sh, &total);
  if (threadIdx.x == 0) cnt[blockIdx.x] = total;
}

// cnt[0..nblk) -> exclusive prefix sums; *pool_rows = 1 + the total
__global__ void __launch_bounds__(1024) rec_pool_scan_kernel(int* __restrict__ cnt, int nblk, int* __restrict__ pool_rows) {
  __shared__ int sh[33];
  int carry = 0;
  for (int i0 = 0; i0 < nblk; i0 += 1024) {
    const int i = i0 + (int)threadIdx.x;
    const int v = i < nblk ? cnt[i] : 0;
    int total;
    const int e = block_scan_excl(v, sh, &total);
    if (i < nblk) cnt[i] = carry + e;
    carry += total;
  }
  if (threadIdx.x == 0) *pool_rows = 1 + carry;
}

__global__ void __launch_bounds__(256) rec_pool_write_kernel(const uint8_t* __restrict__ mask, long long n_rows,
                                                             const int* __restrict__ offs, const uint8_t* __restrict__ cat,
                                                             int32_t* __restrict__ ids, uint8_t* __restrict__ pcat) {
  __shared__ int sh[33];
  const long long r0 = (long long)blockIdx.x * RP_ROWS + 4 * threadIdx.x;
  const int f = pool_flags(mask, n_rows, r0);
  int total;
  int o = 1 + offs[blockIdx.x] + block_scan_excl(__popc(f), sh, &total);
#pragma unroll
  for (int q = 0; q < 4; ++q)
    if (f & (1 << q)) {
      ids[o] = (int32_t)(r0 + q);
      if (pcat != nullptr) pcat[o] = cat[r0 + q];
      ++o;
    }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    ids[0] = 0;
    if (pcat != nullptr) pcat[0] = 0;
  }
}

// -------------------------------------------------------------------------------------------- stage 1 (tensor cores)
struct RsParams {
  RecWs w;
  long long n_rows;
  int B, D, S, tiles_per_slice, n_tiles, n_utiles, k, P;
  const uint8_t* cat;                  // [n_rows] category of each row (NULL: no category filter)
  const unsigned long long* ucat;      // [B] allowed categories of each user, bit c for category c
};

// The warp compacts lane L's list: row 0 and the rows of its exclusion list `ex` (nx ascending ids: the user's
// exclusions inside the slice) are dropped; theta = the k-th best t of the rest (the largest order key K with #{keys >= K} >= k, by bisection
// over the 32 key bits; entries are held 16 per lane), and rows below theta - 2 eps are dropped too, in order.
// Returns the new length to every lane; `thr` of lane L becomes theta - 2 eps once there are k rows left.
__device__ __forceinline__ int rs_compact(int L, int2* list_l, const int* ex_l, int nx_l, int cnt_l, int k, float eps2_l,
                                          float& thr) {
  const int lane = threadIdx.x & 31;
  const int n = __shfl_sync(0xffffffffu, cnt_l, L);
  const float e2 = __shfl_sync(0xffffffffu, eps2_l, L);
  int2* list = reinterpret_cast<int2*>(__shfl_sync(0xffffffffu, (unsigned long long)list_l, L));
  const int* ex = reinterpret_cast<const int*>(__shfl_sync(0xffffffffu, (unsigned long long)ex_l, L));
  const int nx = __shfl_sync(0xffffffffu, nx_l, L);
  if (n < k) return n;                                   // no k-th best yet: nothing can be dropped
  const int xv = lane < nx ? __ldg(ex + lane) : 0;       // up to 32 exclusions, loaded with the entries
  int2 e[RS_CAP / 32];
#pragma unroll
  for (int i = 0; i < RS_CAP / 32; ++i) {
    const int j = lane + 32 * i;
    e[i] = j < n ? list[j] : make_int2(0, 0);            // past the end: row 0, dropped
  }
  bool drop[RS_CAP / 32];
#pragma unroll
  for (int i = 0; i < RS_CAP / 32; ++i) drop[i] = e[i].y == 0;
  if (nx <= 32) {                                        // the usual case: compare with each exclusion in turn
    for (int q = 0; q < nx; ++q) {
      const int v = __shfl_sync(0xffffffffu, xv, q);
#pragma unroll
      for (int i = 0; i < RS_CAP / 32; ++i) drop[i] |= e[i].y == v;
    }
  } else {                                               // many: binary search per entry
    int lo[RS_CAP / 32];
#pragma unroll
    for (int i = 0; i < RS_CAP / 32; ++i) lo[i] = 0;
    for (int step = 1 << (31 - __clz(nx)); step > 0; step >>= 1)
#pragma unroll
      for (int i = 0; i < RS_CAP / 32; ++i)
        if (lo[i] + step < nx && __ldg(ex + lo[i] + step) <= e[i].y) lo[i] += step;
#pragma unroll
    for (int i = 0; i < RS_CAP / 32; ++i) drop[i] |= __ldg(ex + lo[i]) == e[i].y;
  }
  uint32_t key[RS_CAP / 32];                             // 0: dropped
#pragma unroll
  for (int i = 0; i < RS_CAP / 32; ++i) key[i] = drop[i] ? 0u : order_key(__int_as_float(e[i].x));
  uint32_t K = 0;
  for (int bit = 31; bit >= 0; --bit) {
    const uint32_t c = K | (1u << bit);
    int m = 0;
#pragma unroll
    for (int i = 0; i < RS_CAP / 32; ++i) m += key[i] >= c ? 1 : 0;
    m = __reduce_add_sync(0xffffffffu, m);
    if (m >= k) K = c;
  }
  const float th = K != 0 ? key_to_float(K) - e2 : -INFINITY;   // K = 0: fewer than k rows left, keep them all
  int w = 0;
#pragma unroll
  for (int i = 0; i < RS_CAP / 32; ++i) {
    const bool keep = key[i] != 0 && __int_as_float(e[i].x) >= th;
    const unsigned bal = __ballot_sync(0xffffffffu, keep);
    if (keep) list[w + __popc(bal & ((1u << lane) - 1u))] = e[i];
    w += __popc(bal);
  }
  if (lane == L && K != 0) thr = th;
  return w;
}

// #{i : a[i] < x} of a[0..P) ascending, P a power of two
__device__ __forceinline__ int lower_bound_pow2(const int* a, int P, int x) {
  int lo = 0;
  for (int step = P; step > 0; step >>= 1)
    if (lo + step <= P && a[lo + step - 1] < x) lo += step;
  return lo;
}

__global__ void __launch_bounds__(RS_THREADS, 1)
rec_select_kernel(const __grid_constant__ CUtensorMap tmap_user, const __grid_constant__ CUtensorMap tmap_table,
                  const RsParams p) {
  using namespace gemm;
  extern __shared__ uint8_t rs_smem_raw[];
  const int D = p.D, NKB = D / RS_KB;
  const uint32_t smem_base = (smem_u32(rs_smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = rs_smem_raw + (smem_base - smem_u32(rs_smem_raw));
  // [users: NKB k-blocks of 16 KB][table ring: STAGES x 16 KB][barriers][tmem slot]
  const uint32_t sA = smem_base;
  const uint32_t sB = sA + (uint32_t)NKB * RS_BOX_BYTES;
  const uint32_t bar_base = sB + RS_STAGES * RS_BOX_BYTES;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };                         // leader: both CTAs' table bytes
  auto empty_bar = [&](int s) { return bar_base + 8u * (RS_STAGES + s); };          // each CTA: MMA commit (multicast)
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * RS_STAGES + a); };      // each CTA: MMA commit (multicast)
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * RS_STAGES + 2 + a); }; // leader: both CTAs' epilogue warps
  const uint32_t afull_bar = bar_base + 8u * (2 * RS_STAGES + 4);                   // leader: both CTAs' user bytes
  const uint32_t aempty_bar = bar_base + 8u * (2 * RS_STAGES + 5);                  // each CTA: last MMA of an item
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem_gen + (size_t)(NKB + RS_STAGES) * RS_BOX_BYTES + RS_NBARS * 8);
  const int warp = uniform_warp_id(), lane = threadIdx.x & 31;
  const uint32_t cta_rank = cluster_ctarank();
  const int n_items = p.S * p.n_utiles;                   // item = slice * n_utiles + user tile (slice-major)
  const int i_first = (int)(blockIdx.x >> 1), i_stride = (int)(gridDim.x >> 1);

  if (warp == 4 && lane == 0) {
    for (int s = 0; s < RS_STAGES; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), 2 * 4); }
    mbar_init(afull_bar, 1);
    mbar_init(aempty_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 5) {
    if (lane == 0) { tma_prefetch_desc(&tmap_user); tma_prefetch_desc(&tmap_table); }
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(512)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  auto slice_tiles = [&](int slice, int& t0, int& t1) {
    t0 = slice * p.tiles_per_slice;
    t1 = min(p.n_tiles, t0 + p.tiles_per_slice);
  };

  if (warp == 5) {
    // ===================== TMA producer: the item's 128 users of this CTA, then its table rows k-block by k-block =====
    int stage = 0, it = 0;
    uint32_t phase = 0;
    const uint32_t fb_a = mapa_cluster(afull_bar, 0);
    for (int item = i_first; item < n_items; item += i_stride, ++it) {
      const int slice = item / p.n_utiles, ut = item - slice * p.n_utiles;
      int t0, t1;
      slice_tiles(slice, t0, t1);
      mbar_wait(aempty_bar, ((uint32_t)it & 1u) ^ 1u);   // the previous item's MMAs have read the users
      if (elect_one()) {
        if (cta_rank == 0) mbar_expect_tx(afull_bar, 2u * NKB * RS_BOX_BYTES);
        for (int kb = 0; kb < NKB; ++kb)
          tma_load_2d_cta2(sA + kb * RS_BOX_BYTES, &tmap_user, fb_a, kb * RS_KB, ut * 2 * RS_ROWS + (int)cta_rank * RS_ROWS);
      }
      __syncwarp();
      for (int tile = t0; tile < t1; ++tile)
        for (int kb = 0; kb < NKB; ++kb) {
          mbar_wait(empty_bar(stage), phase ^ 1u);
          if (elect_one()) {
            if (cta_rank == 0) mbar_expect_tx(full_bar(stage), 2u * RS_BOX_BYTES);
            tma_load_2d_cta2(sB + stage * RS_BOX_BYTES, &tmap_table, mapa_cluster(full_bar(stage), 0), kb * RS_KB,
                             tile * RS_TN + (int)cta_rank * (RS_TN / 2));
          }
          __syncwarp();
          if (++stage == RS_STAGES) { stage = 0; phase ^= 1u; }
        }
    }
  } else if (warp == 4) {
    // ===================== MMA issuer: the leader's warp walks the loop, one elected lane issues =====================
    if (cta_rank == 0) {
      // D f32, A / B tf32 K-major, N = 256 table rows, M = 256 users across the pair
      constexpr uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(RS_TN >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
      const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
      int stage = 0, acc = 0, it = 0;
      uint32_t phase = 0, acc_phase = 0;
      for (int item = i_first; item < n_items; item += i_stride, ++it) {
        int t0, t1;
        slice_tiles(item / p.n_utiles, t0, t1);
        mbar_wait(afull_bar, (uint32_t)it & 1u);
        for (int tile = t0; tile < t1; ++tile) {
          mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
          tc_fence_after();
          const uint32_t tmem_d = tmem_u + (uint32_t)(acc * RS_TN);
          for (int kb = 0; kb < NKB; ++kb) {
            mbar_wait(full_bar(stage), phase);
            tc_fence_after();
            const uint64_t adesc = make_desc_kmajor_sw128(sA + (uint32_t)kb * RS_BOX_BYTES);
            const uint64_t bdesc = make_desc_kmajor_sw128(sB + (uint32_t)stage * RS_BOX_BYTES);
            if (elect_one()) {
#pragma unroll
              for (int k = 0; k < RS_KB / 8; ++k)          // kind::tf32: K = 8 per instruction, +32 B inside the atom
                tc_mma_tf32_cta2(tmem_d, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (kb > 0 || k > 0) ? 1u : 0u);
              tc_commit_mc2(empty_bar(stage), 3);
            }
            __syncwarp();
            if (++stage == RS_STAGES) { stage = 0; phase ^= 1u; }
          }
          if (elect_one()) tc_commit_mc2(tfull_bar(acc), 3);
          __syncwarp();
          acc ^= 1; if (acc == 0) acc_phase ^= 1u;
        }
        if (elect_one()) tc_commit_mc2(aempty_bar, 3);     // both CTAs may load the next item's users
        __syncwarp();
      }
    }
  } else {
    // ===================== epilogue: a thread owns a user (TMEM lane), a list per (user, slice) =====================
    const int quarter = warp;
    const uint32_t tempty_remote = mapa_cluster(tempty_bar(0), 0);
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int item = i_first; item < n_items; item += i_stride) {
      const int slice = item / p.n_utiles, ut = item - slice * p.n_utiles;
      int t0, t1;
      slice_tiles(slice, t0, t1);
      const int b = ut * 2 * RS_ROWS + (int)cta_rank * RS_ROWS + quarter * 32 + lane;
      const bool valid = b < p.B;
      const float eps2 = valid ? p.w.eps2[b] : 0.f;
      const unsigned long long cmask = valid && p.ucat != nullptr ? p.ucat[b] : ~0ull;
      int2* list = p.w.lists + ((size_t)slice * p.B + (valid ? b : 0)) * RS_CAP;
      // the user's exclusions inside the slice's rows (ascending): the only ones its list can hold
      const int* ex = p.w.excl + (size_t)(valid ? b : 0) * p.P;
      int nx = 0;
      if (valid && p.P > 0) {
        const int e0 = lower_bound_pow2(ex, p.P, t0 * RS_TN);
        nx = lower_bound_pow2(ex, p.P, t1 * RS_TN) - e0;
        ex += e0;
      }
      int cnt = valid ? 0 : RS_CAP + 1;                   // > RS_CAP: appends off (overflowed, or no user)
      float thr = -INFINITY;
      for (int tile = t0; tile < t1; ++tile) {
        mbar_wait(tfull_bar(acc), acc_phase);
        tc_fence_after();
        const uint32_t t_row = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * RS_TN);
        uint32_t ra[32], rb[32];
        tmem_ld32(t_row, ra);
        auto chunk = [&](const uint32_t (&r)[32], int c0) {
          // room for a whole chunk first: lists about to fill are compacted by their warp, one lane at a time
          unsigned need = __ballot_sync(0xffffffffu, cnt <= RS_CAP && cnt > RS_CAP - 32);
          while (need) {
            const int L = __ffs(need) - 1;
            need &= need - 1;
            const int w = rs_compact(L, list, ex, nx, cnt, p.k, eps2, thr);
            if (lane == L) cnt = w > RS_CAP - 32 ? RS_CAP + 1 : w;
          }
          float mx = -INFINITY;
#pragma unroll
          for (int j = 0; j < 32; ++j) mx = fmaxf(mx, __uint_as_float(r[j]));
          const bool on = cnt <= RS_CAP && mx >= thr;
          if (__any_sync(0xffffffffu, on) && on) {
            const long long row0 = (long long)tile * RS_TN + c0;
            const int lim = (int)min(32LL, p.n_rows - row0);       // the last tile's columns past the table are zero
            if (p.cat == nullptr) {
#pragma unroll
              for (int j = 0; j < 32; ++j) {
                const float t = __uint_as_float(r[j]);
                if (j < lim && t >= thr) list[cnt++] = make_int2(__float_as_int(t), (int)row0 + j);
              }
            } else {
#pragma unroll
              for (int j = 0; j < 32; ++j) {
                const float t = __uint_as_float(r[j]);
                // only rows past the threshold read their category: the same byte for the whole warp (a broadcast)
                if (j < lim && t >= thr && ((cmask >> (__ldg(p.cat + row0 + j) & 63)) & 1ull))
                  list[cnt++] = make_int2(__float_as_int(t), (int)row0 + j);
              }
            }
          }
        };
#pragma unroll
        for (int c0 = 0; c0 < RS_TN; c0 += 64) {
          tmem_ld_wait();
          tmem_ld32(t_row + (uint32_t)(c0 + 32), rb);
          chunk(ra, c0);
          tmem_ld_wait();
          if (c0 + 64 < RS_TN) tmem_ld32(t_row + (uint32_t)(c0 + 64), ra);
          else {
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(tempty_remote + 8u * acc);   // the accumulator stage is in registers
          }
          chunk(rb, c0 + 32);
        }
        acc ^= 1; if (acc == 0) acc_phase ^= 1u;
      }
      // the slice is done: shrink every list to its final theta (fewer rows for stage 2)
      unsigned need = __ballot_sync(0xffffffffu, cnt <= RS_CAP && cnt > p.k);
      while (need) {
        const int L = __ffs(need) - 1;
        need &= need - 1;
        const int w = rs_compact(L, list, ex, nx, cnt, p.k, eps2, thr);
        if (lane == L) cnt = w;
      }
      if (valid) p.w.cnt[(size_t)slice * p.B + b] = cnt;
    }
  }

  tc_fence_before();
  cluster_sync_all();
  if (warp == 5)
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(512) : "memory");
}

// ---------------------------------------------------------------------------------------- block-wide exact selection
// The k-th largest of the keys s[0..n) (1 <= k <= n): an 8-bit radix select from the top byte.  hist: 258 ints.
__device__ uint64_t block_kth_largest(const uint64_t* s, int n, int k, int* hist) {
  uint64_t prefix = 0, mask = 0;
  int kk = k;
  for (int shift = 56; shift >= 0; shift -= 8) {
    for (int i = threadIdx.x; i < 256; i += blockDim.x) hist[i] = 0;
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      const uint64_t key = s[i];
      if ((key & mask) == prefix) atomicAdd(&hist[(int)(key >> shift) & 255], 1);
    }
    __syncthreads();
    if (threadIdx.x < 32) {
      const int l = threadIdx.x;
      int c = 0;
#pragma unroll
      for (int j = 0; j < 8; ++j) c += hist[8 * l + j];
      int suf = c;                                       // keys in the bins of lanes >= l
      for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_down_sync(0xffffffffu, suf, o);
        if (l + o < 32) suf += v;
      }
      if (suf - c < kk && suf >= kk) {
        int a = suf - c, d = 8 * l + 7;
        while (a + hist[d] < kk) { a += hist[d]; --d; }
        hist[256] = d;
        hist[257] = a;
      }
    }
    __syncthreads();
    prefix |= (uint64_t)hist[256] << shift;
    mask |= (uint64_t)0xff << shift;
    kk -= hist[257];
    __syncthreads();
  }
  return prefix;
}

// The k largest of s[0..n) (k <= n), descending, into dst[0..k).  tmp: k keys; hist: 259 ints.
__device__ void block_topk(const uint64_t* s, int n, int k, int* hist, uint64_t* tmp, uint64_t* dst) {
  const uint64_t K = block_kth_largest(s, n, k, hist);
  if (threadIdx.x == 0) hist[258] = 0;
  __syncthreads();
  for (int i = threadIdx.x; i < n; i += blockDim.x)
    if (s[i] > K) tmp[atomicAdd(&hist[258], 1)] = s[i];
  __syncthreads();
  for (int i = hist[258] + (int)threadIdx.x; i < k; i += blockDim.x) tmp[i] = K;   // K itself (and equal zero keys)
  __syncthreads();
  for (int i = threadIdx.x; i < k; i += blockDim.x) {
    const uint64_t v = tmp[i];
    int r = 0;
    for (int j = 0; j < k; ++j) r += (tmp[j] > v || (tmp[j] == v && j < i)) ? 1 : 0;
    dst[r] = v;
  }
  __syncthreads();
}

__device__ __forceinline__ bool excluded(const int* ex, int P, int row) {   // ex ascending, P a power of two (or 0)
  if (P == 0) return false;
  int lo = 0;
  for (int step = P >> 1; step > 0; step >>= 1)
    if (ex[lo + step] <= row) lo += step;
  return ex[lo] == row;
}

// map: table id of each local row (NULL: the identity)
__device__ void write_result(const uint64_t* dst, int k, int b, const int32_t* map, int32_t* out_idx, float* out_score) {
  for (int i = threadIdx.x; i < k; i += blockDim.x) {
    const uint64_t key = dst[i];
    const int32_t row = (int32_t)(0xffffffffu - (uint32_t)key);
    // eval_dot8 never returns -0 (the sums start at +0), so the key gives back the score's bits
    out_idx[(size_t)b * k + i] = key ? (map != nullptr ? map[row] : row) : -1;
    out_score[(size_t)b * k + i] = key ? key_to_float((uint32_t)(key >> 32)) : -INFINITY;
  }
}

// eval scores of rows[0..n) for user u: keys[i] = rank_key(s, row); an 8-lane group per row, four rows per warp pass
template <int VPL>
__device__ void score_rows(const float* __restrict__ table, const float* __restrict__ u, const int* rows, int n,
                           uint64_t* keys) {
  const int lane = threadIdx.x & 31, grp = lane >> 3, gl = lane & 7, warp = threadIdx.x >> 5;
  const int nw = blockDim.x >> 5;
  constexpr int D = 32 * VPL;
  float4 uu[VPL];
#pragma unroll
  for (int v = 0; v < VPL; ++v) uu[v] = __ldg(reinterpret_cast<const float4*>(u) + gl + v * 8);
  for (int i0 = warp * 4; i0 < n; i0 += nw * 4) {
    const int i = i0 + grp;
    const bool live = i < n;
    const int row = live ? rows[i] : 0;
    const float4* xr = reinterpret_cast<const float4*>(table + (size_t)row * D) + gl;
    float4 x[VPL];
#pragma unroll
    for (int v = 0; v < VPL; ++v) x[v] = live ? __ldg(xr + v * 8) : make_float4(0.f, 0.f, 0.f, 0.f);
    const float s = eval_dot8<VPL>(x, uu);
    if (live && gl == 0) keys[i] = rank_key(s, row);
  }
}

// ------------------------------------------------------------------------------------------------ stage 2 (exact merge)
struct RmParams {
  RecWs w;
  const float* table;
  const float* user;
  const int32_t* map;                  // [n_rows] table id of each local row (NULL: the identity)
  const uint8_t* cat;                  // as RsParams
  const unsigned long long* ucat;
  long long n_rows;
  int32_t* out_idx;
  float* out_score;
  int32_t* info;
  int B, S, P, k;
};

template <int VPL>
__global__ void __launch_bounds__(RM_THREADS) rec_merge_kernel(const RmParams p) {
  extern __shared__ __align__(16) uint8_t rm_smem[];
  uint64_t* keys = reinterpret_cast<uint64_t*>(rm_smem);                // [RM_UCAP]
  int* rows = reinterpret_cast<int*>(keys + RM_UCAP);                   // [RM_UCAP]
  int* ex = rows + RM_UCAP;                                             // [P]
  uint64_t* tmp = reinterpret_cast<uint64_t*>(ex + ((p.P + 1) & ~1));   // [64]
  uint64_t* dst = tmp + 64;                                             // [64]
  __shared__ int hist[260];
  __shared__ int offs[RS_MAX_SLICES + 1];
  const int b = blockIdx.x, t = threadIdx.x;
  if (t == 0) {
    int o = 0;
    bool over = false;
    for (int s = 0; s < p.S; ++s) {
      const int c = p.w.cnt[(size_t)s * p.B + b];
      over |= c > RS_CAP;
      offs[s] = o;
      o += c;
    }
    offs[p.S] = (over || o > RM_UCAP) ? -1 : o;
    if (offs[p.S] < 0) {
      p.w.fb[atomicAdd(reinterpret_cast<int*>(p.w.hdr) + 1, 1)] = b;
      p.info[1 + b] = -1;
    }
  }
  __syncthreads();
  const int n_u = offs[p.S];
  if (n_u < 0) return;                                   // the exact pass takes this user
  for (int i = t; i < p.P; i += RM_THREADS) ex[i] = p.w.excl[(size_t)b * p.P + i];
  __syncthreads();
  for (int s = 0; s < p.S; ++s) {
    const int2* list = p.w.lists + ((size_t)s * p.B + b) * RS_CAP;
    const int c = (s + 1 < p.S ? offs[s + 1] : n_u) - offs[s];
    for (int j = t; j < c; j += RM_THREADS) {
      const int2 e = list[j];
      const bool ok = e.y >= 1 && !excluded(ex, p.P, e.y);
      keys[offs[s] + j] = ok ? rank_key(__int_as_float(e.x), e.y) : 0ull;
    }
  }
  if (t == 0) hist[259] = 0;
  __syncthreads();
  int ne = 0;
  for (int i = t; i < n_u; i += RM_THREADS) ne += keys[i] != 0ull;
  atomicAdd(&hist[259], ne);
  __syncthreads();
  const int n_e = hist[259];
  __syncthreads();
  if (t == 0) p.info[1 + b] = n_e;
  float thr = -INFINITY;
  if (n_e > p.k) thr = key_to_float((uint32_t)(block_kth_largest(keys, n_u, p.k, hist) >> 32)) - p.w.eps2[b];
  if (t == 0) hist[259] = 0;
  __syncthreads();
  for (int i = t; i < n_u; i += RM_THREADS) {
    const uint64_t key = keys[i];
    if (key != 0ull && key_to_float((uint32_t)(key >> 32)) >= thr)
      rows[atomicAdd(&hist[259], 1)] = (int)(0xffffffffu - (uint32_t)key);
  }
  __syncthreads();
  const int n_s = hist[259];
  score_rows<VPL>(p.table, p.user + (size_t)b * 32 * VPL, rows, n_s, keys);
  __syncthreads();
  for (int i = n_s + t; i < p.k; i += RM_THREADS) keys[i] = 0ull;
  __syncthreads();
  block_topk(keys, max(n_s, p.k), p.k, hist, tmp, dst);
  write_result(dst, p.k, b, p.map, p.out_idx, p.out_score);
}

// ---------------------------------------------------------------------------- fallback: every eligible row, exactly
template <int VPL>
__global__ void __launch_bounds__(RM_THREADS, 1) rec_exact_kernel(const RmParams p) {
  extern __shared__ __align__(16) uint8_t rx_smem[];
  uint64_t* keys = reinterpret_cast<uint64_t*>(rx_smem);                // [64 + RX_CHUNK]: running top k, then a chunk
  int* rows = reinterpret_cast<int*>(keys + 64 + RX_CHUNK);             // [RX_CHUNK]
  int* ex = rows + RX_CHUNK;                                            // [P]
  uint64_t* tmp = reinterpret_cast<uint64_t*>(ex + ((p.P + 1) & ~1));
  __shared__ int hist[260];
  __shared__ unsigned long long cmask;                                  // the user's allowed categories
  __shared__ int n_fb;
  if (threadIdx.x == 0) n_fb = reinterpret_cast<const int*>(p.w.hdr)[1];
  __syncthreads();
  const int k = p.k;
  for (int f = blockIdx.x; f < n_fb; f += gridDim.x) {
    const int b = p.w.fb[f];
    if (threadIdx.x == 0) cmask = p.ucat != nullptr ? p.ucat[b] : ~0ull;
    for (int i = threadIdx.x; i < p.P; i += RM_THREADS) ex[i] = p.w.excl[(size_t)b * p.P + i];
    for (int i = threadIdx.x; i < k; i += RM_THREADS) keys[i] = 0ull;
    __syncthreads();
    for (long long r0 = 1; r0 < p.n_rows; r0 += RX_CHUNK) {
      if (threadIdx.x == 0) hist[259] = 0;
      __syncthreads();
      for (int i = threadIdx.x; i < RX_CHUNK; i += RM_THREADS) {
        const long long r = r0 + i;
        const int rr = r < p.n_rows ? (int)r : 0;                   // row 0: never eligible
        bool ok = rr != 0 && !excluded(ex, p.P, rr);
        if (p.cat != nullptr) ok = ok && ((cmask >> (p.cat[rr] & 63)) & 1ull) != 0;
        const unsigned bal = __ballot_sync(0xffffffffu, ok);
        int base = 0;
        if ((threadIdx.x & 31) == 0 && bal) base = atomicAdd(&hist[259], __popc(bal));
        base = __shfl_sync(0xffffffffu, base, 0);
        if (ok) rows[base + __popc(bal & ((1u << (threadIdx.x & 31)) - 1u))] = (int)r;
      }
      __syncthreads();
      const int n = hist[259];
      score_rows<VPL>(p.table, p.user + (size_t)b * 32 * VPL, rows, n, keys + k);
      __syncthreads();
      block_topk(keys, k + n, k, hist, tmp, tmp + 64);
      for (int i = threadIdx.x; i < k; i += RM_THREADS) keys[i] = tmp[64 + i];
      __syncthreads();
    }
    write_result(keys, k, b, p.map, p.out_idx, p.out_score);
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------------------------------- host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// fp32 [outer, D] row-major -> boxes of 128 rows x 32 floats, 128B-swizzled (the K-major UMMA operand layout); rows past
// `outer` read as zeros
static int make_map_f32(CUtensorMap* map, const float* ptr, int D, long long outer) {
  static EncodeTiledFn enc = nullptr;
  if (enc == nullptr) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      enc = reinterpret_cast<EncodeTiledFn>(fn);
  }
  TNR_REQUIRE(enc != nullptr, "cuTensorMapEncodeTiled driver entry point not available");
  cuuint64_t dims[2] = {(cuuint64_t)D, (cuuint64_t)outer};
  cuuint64_t strides[1] = {(cuuint64_t)D * 4};
  cuuint32_t box[2] = {RS_KB, 128};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(ptr), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  TNR_REQUIRE(r == CUDA_SUCCESS, "tnr_recommend: cuTensorMapEncodeTiled failed (CUresult %d)", (int)r);
  return 0;
}

// The optional filters of a call (all NULL / 0: the unfiltered call)
struct RecFilters {
  const int32_t* excl;                 // [B, E] listed ids per user (table ids)
  int E;
  const int32_t* map;                  // [n_rows] ascending table ids of the pool's rows, map[0] = 0 (NULL: no pool)
  const uint8_t* cat;                  // [n_rows] category (< 64) of each row scored
  const unsigned long long* ucat;      // [B] allowed categories of each user
};

static int rec_check(const char* who, const float* table, long long n_rows, const float* user, int B, int D, int H, int k,
                     void* ws, long long ws_bytes, int exclude, const RecFilters& f) {
  TNR_REQUIRE(k >= 1 && k <= 64, "%s: k=%d must be in 1..64", who, k);
  TNR_REQUIRE(D % 32 == 0 && D >= 32 && D <= RS_DMAX, "%s: D=%d must be a multiple of 32 in 32..256", who, D);
  TNR_REQUIRE(H >= 1 && H <= 512, "%s: H=%d must be in 1..512", who, H);
  TNR_REQUIRE(f.E >= 0 && f.E <= RS_MAX_EXCL - 512, "%s: E=%d must be in 0..512", who, f.E);
  TNR_REQUIRE((f.cat == nullptr) == (f.ucat == nullptr), "%s: category and user_categories go together", who);
  TNR_REQUIRE(B >= 0 && n_rows >= 1 && n_rows < (1LL << 31) - RS_TN, "%s: B=%d / n_rows=%lld out of range", who, B, n_rows);
  TNR_REQUIRE(table != nullptr && user != nullptr && (uintptr_t)table % 16 == 0 && (uintptr_t)user % 16 == 0,
              "%s: table and user must be 16-byte aligned device arrays", who);
  const RecShape s = rec_shape(n_rows, B, H, exclude, f.E);
  TNR_REQUIRE(ws != nullptr && (uintptr_t)ws % 256 == 0 && ws_bytes >= (long long)rec_layout(s, B, nullptr, nullptr),
              "%s: workspace of tnr_recommend_filtered_ws_bytes bytes (256-byte aligned) required", who);
  return 0;
}

template <int VPL>
static int rec_merge_launch(const RmParams& p, cudaStream_t st) {
  const int ex_bytes = ((p.P + 1) & ~1) * 4;
  const int m_smem = RM_UCAP * 12 + ex_bytes + 128 * 8;
  const int x_smem = (64 + RX_CHUNK) * 8 + RX_CHUNK * 4 + ex_bytes + 128 * 8;
  TNR_SET_SMEM(rec_merge_kernel<VPL>, m_smem);
  TNR_SET_SMEM(rec_exact_kernel<VPL>, x_smem);
  if (p.B > 0) rec_merge_kernel<VPL><<<p.B, RM_THREADS, m_smem, st>>>(p);
  TNR_LAUNCH_CHECK();
  const int grid = p.B < 2 * num_sms() ? (p.B > 0 ? p.B : 1) : 2 * num_sms();
  rec_exact_kernel<VPL><<<grid, RM_THREADS, x_smem, st>>>(p);
  TNR_LAUNCH_CHECK();
  return 0;
}

static int rec_select(const char* who, const float* table, long long n_rows, const float* user, int B, int D,
                      const int32_t* hist_idx, const float* hist_mask, int H, int k, int exclude_history,
                      const RecFilters& f, void* workspace, long long ws_bytes, void* stream) {
  if (rec_check(who, table, n_rows, user, B, D, H, k, workspace, ws_bytes, exclude_history, f)) return 1;
  TNR_REQUIRE(!exclude_history || (hist_idx != nullptr && hist_mask != nullptr),
              "%s: the history is required with exclude_history", who);
  TNR_REQUIRE(f.E == 0 || f.excl != nullptr, "%s: the exclusion list is required with E > 0", who);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const RecShape s = rec_shape(n_rows, B, H, exclude_history, f.E);
  RecWs w;
  rec_layout(s, B, reinterpret_cast<char*>(workspace), &w);
  TNR_CHECK_CUDA(cudaMemsetAsync(w.hdr, 0, 16, st));
  if (B == 0) return 0;
  const long long nb = (n_rows + 7) / 8;
  rec_table_norm_kernel<<<(int)(nb < 4 * num_sms() ? nb : 4 * num_sms()), 256, 0, st>>>(table, n_rows, D, w.hdr);
  TNR_LAUNCH_CHECK();
  rec_prep_kernel<<<B, 256, 0, st>>>(user, D, hist_idx, hist_mask, exclude_history ? H : 0, f.excl, f.E, f.map, n_rows,
                                     w, s.P);
  TNR_LAUNCH_CHECK();
  CUtensorMap tu, tt;
  if (make_map_f32(&tu, user, D, B) || make_map_f32(&tt, table, D, n_rows)) return 1;
  RsParams p;
  p.w = w; p.n_rows = n_rows; p.B = B; p.D = D; p.S = s.S; p.tiles_per_slice = s.tiles_per_slice; p.n_tiles = s.n_tiles;
  p.n_utiles = s.n_utiles; p.k = k; p.P = s.P; p.cat = f.cat; p.ucat = f.ucat;
  const int items = s.S * s.n_utiles;
  const int pairs = items < num_sms() / 2 ? items : num_sms() / 2;
  TNR_SET_SMEM(rec_select_kernel, rs_smem_bytes(RS_DMAX));
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2 * pairs);
  cfg.blockDim = dim3(RS_THREADS);
  cfg.dynamicSmemBytes = rs_smem_bytes(D);
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  TNR_CHECK_CUDA(cudaLaunchKernelEx(&cfg, rec_select_kernel, tu, tt, p));
  return 0;
}

static int rec_merge(const char* who, const float* table, long long n_rows, const float* user, int B, int D, int H, int k,
                     int exclude_history, const RecFilters& f, int32_t* out_idx, float* out_score, int32_t* info,
                     void* workspace, long long ws_bytes, void* stream) {
  if (rec_check(who, table, n_rows, user, B, D, H, k, workspace, ws_bytes, exclude_history, f)) return 1;
  TNR_REQUIRE(out_idx != nullptr && out_score != nullptr && info != nullptr,
              "%s: out_idx int32 [B, k], out_score fp32 [B, k] and info int32 [B + 1] are required", who);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const RecShape s = rec_shape(n_rows, B, H, exclude_history, f.E);
  RmParams p;
  rec_layout(s, B, reinterpret_cast<char*>(workspace), &p.w);
  p.table = table; p.user = user; p.map = f.map; p.cat = f.cat; p.ucat = f.ucat; p.n_rows = n_rows;
  p.out_idx = out_idx; p.out_score = out_score; p.info = info;
  p.B = B; p.S = s.S; p.P = s.P; p.k = k;
  int rc;
  switch (D / 32) {
    case 1: rc = rec_merge_launch<1>(p, st); break;
    case 2: rc = rec_merge_launch<2>(p, st); break;
    case 4: rc = rec_merge_launch<4>(p, st); break;
    case 8: rc = rec_merge_launch<8>(p, st); break;
    default: set_error("%s: D=%d not instantiated (32, 64, 128, 256)", who, D); return 1;
  }
  if (rc) return rc;
  TNR_CHECK_CUDA(cudaMemcpyAsync(info, reinterpret_cast<int*>(p.w.hdr) + 1, 4, cudaMemcpyDeviceToDevice, st));
  return 0;
}

}  // namespace
}  // namespace tnr

using namespace tnr;

TNR_API long long tnr_recommend_ws_bytes(long long n_rows, int B, int H, int exclude_history) {
  if (n_rows < 1 || B < 0 || H < 1) return -1;
  return (long long)rec_layout(rec_shape(n_rows, B, H, exclude_history, 0), B, nullptr, nullptr);
}

TNR_API int tnr_recommend_select(const float* table, long long n_rows, const float* user, int B, int D,
                                 const int32_t* hist_idx, const float* hist_mask, int H, int k, int exclude_history,
                                 void* workspace, long long ws_bytes, void* stream) {
  return rec_select("tnr_recommend_select", table, n_rows, user, B, D, hist_idx, hist_mask, H, k, exclude_history,
                    RecFilters{}, workspace, ws_bytes, stream);
}

TNR_API int tnr_recommend_merge(const float* table, long long n_rows, const float* user, int B, int D, int H, int k,
                                int exclude_history, int32_t* out_idx, float* out_score, int32_t* info, void* workspace,
                                long long ws_bytes, void* stream) {
  return rec_merge("tnr_recommend_merge", table, n_rows, user, B, D, H, k, exclude_history, RecFilters{}, out_idx,
                   out_score, info, workspace, ws_bytes, stream);
}

TNR_API long long tnr_recommend_filtered_ws_bytes(long long n_rows, int B, int H, int exclude_history, int E) {
  if (n_rows < 1 || B < 0 || H < 1 || E < 0 || E > 512) return -1;
  return (long long)rec_layout(rec_shape(n_rows, B, H, exclude_history, E), B, nullptr, nullptr);
}

TNR_API int tnr_recommend_select_filtered(const float* table, long long n_rows, const float* user, int B, int D,
                                          const int32_t* hist_idx, const float* hist_mask, int H, int k,
                                          int exclude_history, const int32_t* exclude, int E, const int32_t* pool_ids,
                                          const uint8_t* category, const unsigned long long* user_categories,
                                          void* workspace, long long ws_bytes, void* stream) {
  return rec_select("tnr_recommend_select_filtered", table, n_rows, user, B, D, hist_idx, hist_mask, H, k,
                    exclude_history, RecFilters{exclude, E, pool_ids, category, user_categories}, workspace, ws_bytes,
                    stream);
}

TNR_API int tnr_recommend_merge_filtered(const float* table, long long n_rows, const float* user, int B, int D, int H,
                                         int k, int exclude_history, int E, const int32_t* pool_ids,
                                         const uint8_t* category, const unsigned long long* user_categories,
                                         int32_t* out_idx, float* out_score, int32_t* info, void* workspace,
                                         long long ws_bytes, void* stream) {
  return rec_merge("tnr_recommend_merge_filtered", table, n_rows, user, B, D, H, k, exclude_history,
                   RecFilters{nullptr, E, pool_ids, category, user_categories}, out_idx, out_score, info, workspace,
                   ws_bytes, stream);
}

TNR_API long long tnr_recommend_pool_ws_bytes(long long n_rows) {
  if (n_rows < 1) return -1;
  return (long long)align256((size_t)((n_rows + RP_ROWS - 1) / RP_ROWS) * 4);
}

TNR_API int tnr_recommend_pool(const uint8_t* mask, long long n_rows, const uint8_t* category, int32_t* pool_ids,
                               uint8_t* pool_category, int32_t* pool_rows, void* workspace, long long ws_bytes,
                               void* stream) {
  TNR_REQUIRE(n_rows >= 1 && n_rows < (1LL << 31) - RS_TN, "tnr_recommend_pool: n_rows=%lld out of range", n_rows);
  TNR_REQUIRE(mask != nullptr && pool_ids != nullptr && pool_rows != nullptr,
              "tnr_recommend_pool: mask, pool_ids and pool_rows are required");
  TNR_REQUIRE((category == nullptr) == (pool_category == nullptr),
              "tnr_recommend_pool: category and pool_category go together");
  TNR_REQUIRE(workspace != nullptr && ws_bytes >= tnr_recommend_pool_ws_bytes(n_rows),
              "tnr_recommend_pool: workspace of tnr_recommend_pool_ws_bytes bytes required");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int nblk = (int)((n_rows + RP_ROWS - 1) / RP_ROWS);
  int* cnt = reinterpret_cast<int*>(workspace);
  rec_pool_count_kernel<<<nblk, 256, 0, st>>>(mask, n_rows, cnt);
  TNR_LAUNCH_CHECK();
  rec_pool_scan_kernel<<<1, 1024, 0, st>>>(cnt, nblk, pool_rows);
  TNR_LAUNCH_CHECK();
  rec_pool_write_kernel<<<nblk, 256, 0, st>>>(mask, n_rows, cnt, category, pool_ids, pool_category);
  TNR_LAUNCH_CHECK();
  return 0;
}
