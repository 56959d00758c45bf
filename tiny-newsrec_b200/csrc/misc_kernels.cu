// Optimiser, dtype casts, batch-assembly gathers and the impression-scoring metrics kernel.
#include "common.cuh"
#include "eval_score.cuh"

#define TNR_API extern "C" __attribute__((visibility("default")))

namespace tnr {

// ---------------------------------------------------------------------------------
// Adam(amsgrad=True) over one flat fp32 parameter buffer (torch.optim.Adam semantics,
// reference Tiny-NewsRec/run.py:134), fused with the bf16 shadow-weight refresh.
//   m = b1 m + (1-b1) g ; v = b2 v + (1-b2) g^2 ; vmax = max(vmax, v)
//   p -= (lr / bc1) * m / (sqrt(vmax) / sqrt(bc2) + eps)
// grad_scale multiplies g first (1/world for a summed all-reduce).
// ---------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
adam_amsgrad_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                    float* __restrict__ vmax, __nv_bfloat16* __restrict__ shadow, long long n, float lr, float b1,
                    float b2, float eps, float bc1, float rsqrt_bc2, float grad_scale, const float* __restrict__ bc_dev) {
  const long long i4 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i4 >= n) return;
  if (bc_dev != nullptr) { bc1 = bc_dev[0]; rsqrt_bc2 = bc_dev[1]; }      // device-resident step (CUDA-graph replay)
  if (i4 + 4 <= n) {
    float4 pp = *reinterpret_cast<float4*>(p + i4);
    const float4 gg = *reinterpret_cast<const float4*>(g + i4);
    float4 mm = *reinterpret_cast<float4*>(m + i4);
    float4 vv = *reinterpret_cast<float4*>(v + i4);
    const bool ams = vmax != nullptr;          // vmax == NULL: plain Adam (torch amsgrad=False), denominator from v
    float4 vx = ams ? *reinterpret_cast<float4*>(vmax + i4) : make_float4(0.f, 0.f, 0.f, 0.f);
    float* P = reinterpret_cast<float*>(&pp);
    const float* G = reinterpret_cast<const float*>(&gg);
    float* Mm = reinterpret_cast<float*>(&mm);
    float* V = reinterpret_cast<float*>(&vv);
    float* VX = reinterpret_cast<float*>(&vx);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float gr = G[k] * grad_scale;
      Mm[k] = b1 * Mm[k] + (1.0f - b1) * gr;
      V[k] = b2 * V[k] + (1.0f - b2) * gr * gr;
      VX[k] = fmaxf(VX[k], V[k]);
      P[k] -= (lr / bc1) * Mm[k] / (sqrtf(VX[k]) * rsqrt_bc2 + eps);
    }
    *reinterpret_cast<float4*>(p + i4) = pp;
    *reinterpret_cast<float4*>(m + i4) = mm;
    *reinterpret_cast<float4*>(v + i4) = vv;
    if (ams) *reinterpret_cast<float4*>(vmax + i4) = vx;
    if (shadow != nullptr) {
      uint2 o;
      o.x = pack_bf16(P[0], P[1]);
      o.y = pack_bf16(P[2], P[3]);
      *reinterpret_cast<uint2*>(shadow + i4) = o;
    }
  } else {
    for (long long i = i4; i < n; ++i) {
      const float gr = g[i] * grad_scale;
      m[i] = b1 * m[i] + (1.0f - b1) * gr;
      v[i] = b2 * v[i] + (1.0f - b2) * gr * gr;
      float vm = v[i];
      if (vmax != nullptr) { vm = fmaxf(vmax[i], v[i]); vmax[i] = vm; }
      p[i] -= (lr / bc1) * m[i] / (sqrtf(vm) * rsqrt_bc2 + eps);
      if (shadow != nullptr) shadow[i] = __float2bfloat16_rn(p[i]);
    }
  }
}

__global__ void __launch_bounds__(256)
cast_f32_bf16_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ y, long long n) {
  const long long i4 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i4 >= n) return;
  if (i4 + 4 <= n && (((uintptr_t)(x + i4) & 15) == 0) && (((uintptr_t)(y + i4) & 7) == 0)) {
    const float4 a = *reinterpret_cast<const float4*>(x + i4);
    uint2 o;
    o.x = pack_bf16(a.x, a.y);
    o.y = pack_bf16(a.z, a.w);
    *reinterpret_cast<uint2*>(y + i4) = o;
  } else {
    for (long long i = i4; i < n && i < i4 + 4; ++i) y[i] = __float2bfloat16_rn(x[i]);
  }
}

// ---------------------------------------------------------------------------------
// batch assembly gathers (reference: Tiny-NewsRec/dataloader.py:131,138 token rows -> LongTensor;
// :142,144 and :295,301 embedding rows).  Bit-exact copies.
//   i32 table rows -> int64 out (the reference converts the int32 news_combined rows with
//   torch.LongTensor);  f32 table rows -> f32 out.  One warp per output row.
// ---------------------------------------------------------------------------------
constexpr int GI_ROWS = 4;          // rows per warp: four index loads, then four row loads, then four stores in flight
__global__ void __launch_bounds__(256)
gather_rows_i32_i64_kernel(const int32_t* __restrict__ table, long long n_rows_table, const int32_t* __restrict__ idx,
                           long long n, int W, int64_t* __restrict__ out) {
  const long long r0 = ((long long)blockIdx.x * 8 + uniform_warp_id()) * GI_ROWS;
  if (r0 >= n) return;
  const int lane = threadIdx.x & 31;
  long long src[GI_ROWS];
#pragma unroll
  for (int k = 0; k < GI_ROWS; ++k) {
    src[k] = r0 + k < n ? idx[r0 + k] : 0;
    if (src[k] < 0 || src[k] >= n_rows_table) src[k] = 0;      // unknown id -> row 0 (dataloader.py:74)
  }
  if ((W & 1) == 0) {
    // two tokens per lane: one 8-byte load, one 16-byte store (the scalar one-row-per-warp version moved 4 + 8 bytes
    // per request and reached 41 % of HBM peak; rows are 2L int32 = 240 B in, 480 B out)
    for (int c = lane; c < (W >> 1); c += 32) {
      int2 v[GI_ROWS];
#pragma unroll
      for (int k = 0; k < GI_ROWS; ++k) v[k] = reinterpret_cast<const int2*>(table + src[k] * W)[c];
#pragma unroll
      for (int k = 0; k < GI_ROWS; ++k)
        if (r0 + k < n) reinterpret_cast<longlong2*>(out + (r0 + k) * W)[c] = make_longlong2((long long)v[k].x, (long long)v[k].y);
    }
  } else {
    for (int k = 0; k < GI_ROWS && r0 + k < n; ++k)
      for (int c = lane; c < W; c += 32) out[(r0 + k) * W + c] = (int64_t)table[src[k] * W + c];
  }
}

__global__ void __launch_bounds__(256)
gather_rows_f32_kernel(const float* __restrict__ table, long long n_rows_table, const int32_t* __restrict__ idx,
                       long long n, int D, float* __restrict__ out, long long out_ld) {
  const long long r = (long long)blockIdx.x * 8 + uniform_warp_id();
  if (r >= n) return;
  long long src = idx[r];
  if (src < 0 || src >= n_rows_table) src = 0;
  const int lane = threadIdx.x & 31;
  const float4* s = reinterpret_cast<const float4*>(table + src * D);
  float4* d = reinterpret_cast<float4*>(out + r * out_ld);
  for (int c = lane; c < D / 4; c += 32) d[c] = s[c];
}

// ---------------------------------------------------------------------------------
// One launch assembles a whole training batch from its index arrays (reference: Tiny-NewsRec/dataloader.py:129-144):
// rows r < n_hist take hist_idx[r], the rest cand_idx[r - n_hist]; job 0 (blockIdx.y) widens the int32 token row to the
// int64 row Model.forward takes, job 1 + i copies teacher i's fp32 embedding row.  Outputs are laid out
// [history rows | candidate rows], i.e. already concatenated the way the encoder / the loss head read them.  Replaces
// ten row-gather launches, eight copies and a cat per step (~90 us of 3-8 us kernels).
// ---------------------------------------------------------------------------------
constexpr int TB_MAX_TEACHERS = 8;
struct TrainBatchGather {
  const int32_t* news; long long n_rows; int W;
  const float* teacher[TB_MAX_TEACHERS]; float* teacher_out[TB_MAX_TEACHERS]; int M, D; long long out_ld;
  const int32_t *hist_idx, *cand_idx; long long n_hist, n_cand;
  long long* tokens_out;
};

__global__ void __launch_bounds__(256)
train_batch_gather_kernel(const __grid_constant__ TrainBatchGather g) {
  const long long r = (long long)blockIdx.x * 8 + uniform_warp_id();
  if (r >= g.n_hist + g.n_cand) return;
  const int lane = threadIdx.x & 31, job = blockIdx.y;
  long long src = r < g.n_hist ? g.hist_idx[r] : g.cand_idx[r - g.n_hist];
  if (src < 0 || src >= g.n_rows) src = 0;                       // unknown id -> row 0 (dataloader.py:74)
  if (job == 0) {
    const int32_t* s = g.news + src * g.W;
    long long* d = g.tokens_out + r * g.W;
    for (int c = lane; c < g.W; c += 32) d[c] = (long long)s[c];
  } else {
    const float4* s = reinterpret_cast<const float4*>(g.teacher[job - 1] + src * g.D);
    float4* d = reinterpret_cast<float4*>(g.teacher_out[job - 1] + r * g.out_ld);
    for (int c = lane; c < g.D / 4; c += 32) d[c] = s[c];
  }
}

// ---------------------------------------------------------------------------------
// doc-sim diagnostic (reference: Tiny-NewsRec/run.py:292-299): sum over sampled pairs (i, j), i != j, of
// cos(table[i], table[j]) = dot / (|a| |b|) in fp32 (np.dot / np.linalg.norm on float32 rows), summed in fp64.
// One warp per pair, eight pairs per block, one fp64 atomic per block.
// ---------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
doc_sim_kernel(const float* __restrict__ table, long long n_rows, const int32_t* __restrict__ pairs, long long n_pairs,
               int D, double* __restrict__ sum_out) {
  __shared__ double s_part[8];
  const int warp = uniform_warp_id(), lane = threadIdx.x & 31;
  const long long pidx = (long long)blockIdx.x * 8 + warp;
  double c = 0.0;
  if (pidx < n_pairs) {
    const long long i = pairs[2 * pidx], j = pairs[2 * pidx + 1];
    if (i != j && i >= 0 && j >= 0 && i < n_rows && j < n_rows) {
      const float4* a = reinterpret_cast<const float4*>(table + i * D);
      const float4* b = reinterpret_cast<const float4*>(table + j * D);
      float dot = 0.f, na = 0.f, nb = 0.f;
      for (int k = lane; k < D / 4; k += 32) {
        const float4 x = a[k], y = b[k];
        dot = fmaf(x.x, y.x, fmaf(x.y, y.y, fmaf(x.z, y.z, fmaf(x.w, y.w, dot))));
        na = fmaf(x.x, x.x, fmaf(x.y, x.y, fmaf(x.z, x.z, fmaf(x.w, x.w, na))));
        nb = fmaf(y.x, y.x, fmaf(y.y, y.y, fmaf(y.z, y.z, fmaf(y.w, y.w, nb))));
      }
      dot = warp_sum(dot); na = warp_sum(na); nb = warp_sum(nb);
      c = (double)(dot / (sqrtf(na) * sqrtf(nb)));
    }
  }
  if (lane == 0) s_part[warp] = c;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
#pragma unroll
    for (int w = 0; w < 8; ++w) t += s_part[w];
    atomicAdd(sum_out, t);
  }
}

// ---------------------------------------------------------------------------------
// impression scoring + ranking metrics (reference: Tiny-NewsRec/run.py:346-361,
// metrics.py:5-23, sklearn roc_auc_score), two kernels:
//   eval_score_kernel  FLAT over all candidates of the batch: score_i = table[cand_i] . user[imp(i)].  An 8-lane
//                      group owns a candidate (its 1 KB row = 8 x 16 B per lane, all in flight together with the
//                      user row of its impression, which comes from L1 / L2: consecutive candidates share it), a warp
//                      four candidates per pass.  No per-impression blocks: impressions run from 2 to 300 candidates,
//                      and the block-per-impression kernel this replaces left the SMs waiting on block barriers and on
//                      the serial metric tail of every block (ncu: 2.7 barrier + 6.9 long-scoreboard stalls per issued
//                      instruction, 20 % of HBM peak).
//   eval_rank_kernel   warp per impression over the scores (L2-resident):  skip if labels constant (run.py:348);
//                      rank_c = 1 + #{s_j > s_c} + #{s_j == s_c, j > c}     (= np.argsort(score)[::-1] order)
//                      AUC = (sum_pos #neg below + 0.5 #neg tied) / (P N);  MRR = sum_pos 1/rank / P
//                      nDCG@k = sum_{pos, rank<=k} 1/log2(rank+1) / sum_{r<=min(k,P)} 1/log2(r+1)   (binary labels)
// out[imp] = {auc, mrr, ndcg5, ndcg10, valid}
// ---------------------------------------------------------------------------------
// 1 / log2(r + 1), r = 1..10: the only discounts nDCG@5 / nDCG@10 ever use (metrics.py:7-9); fp64 log2() on the device
// is a long software routine
__constant__ double c_disc[10] = {1.0, 0.6309297535714575, 0.5, 0.43067655807339306, 0.38685280723454163,
                                  0.3562071871080222, 0.3333333333333333, 0.31546487678572877, 0.3010299956639812,
                                  0.2890648263178879};

constexpr int ES_WARPS = 8;
constexpr int ES_CPW = 32;            // candidates per warp work item (8 passes of 4)

// VPL = float4 per lane of an 8-lane group and row: D = 32 * VPL floats (D = 256 -> 8); D % 32 == 0 required.
template <int VPL>
__global__ void __launch_bounds__(ES_WARPS * 32)
eval_score_kernel(const float* __restrict__ table, long long n_rows, const float* __restrict__ user,
                  const long long* __restrict__ ptr, const int32_t* __restrict__ cand, long long n_imp, long long nnz,
                  float* __restrict__ score) {
  const int lane = threadIdx.x & 31, grp = lane >> 3, gl = lane & 7;
  const long long warp_global = (long long)blockIdx.x * ES_WARPS + uniform_warp_id();
  const long long n_items = (nnz + ES_CPW - 1) / ES_CPW;
  constexpr int D = 32 * VPL;
  for (long long item = warp_global; item < n_items; item += (long long)gridDim.x * ES_WARPS) {
    const long long c0 = item * ES_CPW;
    // lane l: candidate c0 + l -> its table row and its impression (largest b with ptr[b] <= i)
    const long long ci = c0 + lane;
    long long row = 0, imp = 0;
    if (ci < nnz) {
      const long long v = cand[ci];
      row = (v >= 0 && v < n_rows) ? v : 0;                    // unknown id -> row 0 (dataloader.py:74)
      long long lo = 0, hi = n_imp;                            // ptr[lo] <= ci < ptr[hi]
      while (hi - lo > 1) {
        const long long mid = (lo + hi) >> 1;
        if (__ldg(ptr + mid) <= ci) lo = mid; else hi = mid;
      }
      imp = lo;
    }
    float out = 0.f;
#pragma unroll 2
    for (int pass = 0; pass < ES_CPW / 4; ++pass) {
      const int src = pass * 4 + grp;                          // the lane that holds this group's candidate
      const long long r = __shfl_sync(0xffffffffu, row, src);
      const long long b = __shfl_sync(0xffffffffu, imp, src);
      const bool live = c0 + src < nnz;
      const float4* xr = reinterpret_cast<const float4*>(table + r * D) + gl;
      const float4* ur = reinterpret_cast<const float4*>(user + b * D) + gl;
      float4 x[VPL], u[VPL];
#pragma unroll
      for (int v = 0; v < VPL; ++v) x[v] = live ? __ldg(xr + v * 8) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int v = 0; v < VPL; ++v) u[v] = live ? __ldg(ur + v * 8) : make_float4(0.f, 0.f, 0.f, 0.f);
      const float t = eval_dot8<VPL>(x, u);     // the same summation tree for every row and user (eval_score.cuh)
      // hand the score to the lane that owns the candidate: coalesced store of 32 scores at the end
      const float mine = __shfl_sync(0xffffffffu, t, (lane & 3) * 8);   // lane l takes group (l & 3) of pass (l >> 2)
      if ((lane >> 2) == pass) out = mine;
    }
    if (ci < nnz) score[ci] = out;
  }
}

constexpr int ER_WARPS = 4;          // small blocks: an SM picks up new impressions as soon as four are done

__device__ __forceinline__ double shfl_xor_f64(double v, int o) {
  return __hiloint2double(__shfl_xor_sync(0xffffffffu, __double2hiint(v), o), __shfl_xor_sync(0xffffffffu, __double2loint(v), o));
}

// Warp per impression.  Scores become order-preserving uint32 keys (one integer compare per test); the positives are
// compacted into a list and taken 32 at a time: lane = (positive slot, candidate segment) -- with few positives (the
// common case: ~4 of ~37 candidates) each positive is scanned by 32 / slots lanes over interleaved 4-candidate groups,
// every lane counting in registers; the segments meet in a few shuffles.  No pass over the candidates is serial.
// (v1: one positive at a time, two 5-step shuffle reductions each, a dependent shared-memory read per candidate:
// 39 us per 4 096 impressions; v2: a lane per positive scanning all candidates: 19 us, all of it the tail of the few
// impressions with hundreds of candidates, which are single warps.)
__global__ void __launch_bounds__(ER_WARPS * 32)
eval_rank_kernel(const float* __restrict__ score, const long long* __restrict__ ptr, const int8_t* __restrict__ label,
                 long long n_imp, int cap, double* __restrict__ out) {
  extern __shared__ __align__(16) float sm[];
  const int warp = uniform_warp_id(), lane = threadIdx.x & 31;
  const int wpb = blockDim.x >> 5;
  const long long b = (long long)blockIdx.x * wpb + warp;
  if (b >= n_imp) return;
  uint32_t* s_key = reinterpret_cast<uint32_t*>(sm) + (size_t)warp * cap;                  // [cap] order keys of the scores
  int* s_pos = reinterpret_cast<int*>(sm + (size_t)wpb * cap) + (size_t)warp * cap;        // [cap] indices of the positives
  int8_t* s_lab = reinterpret_cast<int8_t*>(sm + (size_t)2 * wpb * cap) + (size_t)warp * cap;
  const long long p0 = ptr[b];
  const int C = (int)(ptr[b + 1] - p0);
  const int C4 = (C + 3) & ~3;                 // padded to whole 4-candidate groups: key 0 ranks below every real score
  for (int c = lane; c < C4; c += 32) {        // (no float maps to key 0), label "positive": no AUC term.  All loads of
    if (c < C) {                               // this loop are independent (the compaction below reads shared memory)
      s_key[c] = order_key(score[p0 + c]);
      s_lab[c] = label[p0 + c];
    } else {
      s_key[c] = 0u;
      s_lab[c] = 1;
    }
  }
  __syncwarp();
  int P = 0;
  for (int c0 = 0; c0 < C; c0 += 32) {
    const int c = c0 + lane;
    const bool pos = c < C && s_lab[c] != 0;
    const unsigned bal = __ballot_sync(0xffffffffu, pos);
    if (pos) s_pos[P + __popc(bal & ((1u << lane) - 1u))] = c;                // index order is kept
    P += __popc(bal);
  }
  __syncwarp();
  const int N = C - P;
  if (P == 0 || N == 0) {                      // run.py:348 -- skipped impression
    if (lane < 5) out[(size_t)b * 5 + lane] = 0.0;
    return;
  }
  long long auc2 = 0;                          // 2 * (#neg below) + (#neg tied), summed over this lane's positives: exact
  double mrr = 0.0, d5 = 0.0, d10 = 0.0;
  const int G4 = C4 >> 2;                      // 4-candidate groups
  for (int k0 = 0; k0 < P; k0 += 32) {
    const int np = min(32, P - k0);            // positives of this round
    int slots = 1;
    while (slots < np) slots <<= 1;            // power of two >= np
    const int nseg = 32 / slots, slot = lane & (slots - 1), seg = lane / slots;
    const bool have = slot < np;
    const int c = have ? s_pos[k0 + slot] : 0;
    const uint32_t kc = have ? s_key[c] : 0xffffffffu;
    int above = 0, lt = 0, eq = 0;
    for (int g = seg; g < G4; g += nseg) {     // lanes of a segment read the same 16 + 4 bytes: broadcasts
      const uint4 k4 = *reinterpret_cast<const uint4*>(s_key + 4 * g);
      const uint32_t l4 = *reinterpret_cast<const uint32_t*>(s_lab + 4 * g);
      const uint32_t kj[4] = {k4.x, k4.y, k4.z, k4.w};
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int neg = ((l4 >> (8 * u)) & 0xffu) == 0u;
        const int gt = kj[u] > kc, e = kj[u] == kc;
        above += gt | (e & (int)(4 * g + u > c));
        lt += neg & (int)(kj[u] < kc);
        eq += neg & e;
      }
    }
    for (int o = slots; o < 32; o <<= 1) {     // the segments of a positive meet
      above += __shfl_xor_sync(0xffffffffu, above, o);
      lt += __shfl_xor_sync(0xffffffffu, lt, o);
      eq += __shfl_xor_sync(0xffffffffu, eq, o);
    }
    if (have && seg == 0) {
      const int rank = above + 1;
      auc2 += 2 * lt + eq;
      mrr += 1.0 / (double)rank;
      if (rank <= 10) {
        const double disc = c_disc[rank - 1];
        if (rank <= 5) d5 += disc;
        d10 += disc;
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {           // fixed butterfly: the same sums on every run
    auc2 += __shfl_xor_sync(0xffffffffu, auc2, o);
    mrr += shfl_xor_f64(mrr, o);
    d5 += shfl_xor_f64(d5, o);
    d10 += shfl_xor_f64(d10, o);
  }
  if (lane == 0) {
    double i5 = 0.0, i10 = 0.0;
    for (int r = 1; r <= min(P, 10); ++r) {
      const double disc = c_disc[r - 1];
      if (r <= 5) i5 += disc;
      i10 += disc;
    }
    out[(size_t)b * 5 + 0] = 0.5 * (double)auc2 / ((double)P * (double)N);
    out[(size_t)b * 5 + 1] = mrr / (double)P;
    out[(size_t)b * 5 + 2] = d5 / i5;
    out[(size_t)b * 5 + 3] = d10 / i10;
    out[(size_t)b * 5 + 4] = 1.0;
  }
}

// sums[0..3] += metric sums over impressions, sums[4] += number of valid impressions
__global__ void __launch_bounds__(256)
eval_reduce_kernel(const double* __restrict__ per_imp, long long n, double* __restrict__ sums) {
  double acc[5] = {0, 0, 0, 0, 0};
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
#pragma unroll
    for (int k = 0; k < 5; ++k) acc[k] += per_imp[i * 5 + k];
#pragma unroll
  for (int k = 0; k < 5; ++k) {
    double v = acc[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) atomicAdd(sums + k, v);
  }
}

__global__ void __launch_bounds__(256)
dropout_mask_kernel(const tnr_dropout drop, long long n, unsigned char* __restrict__ keep) {
  const DropCfg dc = load_drop(drop);
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (g * 8 >= n) return;
  const uint32_t m = dc.thr16 != 0 ? dropout_keep8(dc, (uint64_t)g) : 0xffu;
  for (int e = 0; e < 8 && g * 8 + e < n; ++e) keep[g * 8 + e] = (m >> e) & 1u;
}

}  // namespace tnr

using namespace tnr;

TNR_API int tnr_dropout_mask(const tnr_dropout* drop, long long n, unsigned char* keep, void* stream) {
  if (n == 0) return 0;
  const long long groups = (n + 7) / 8;
  dropout_mask_kernel<<<(int)((groups + 255) / 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(drop_or_none(drop), n, keep);
  TNR_LAUNCH_CHECK();
  return 0;
}

TNR_API int tnr_adam_amsgrad(float* p, const float* g, float* m, float* v, float* vmax, void* shadow_bf16, long long n,
                             float lr, float beta1, float beta2, float eps, int step, float grad_scale, void* stream) {
  TNR_REQUIRE(step >= 1, "tnr_adam_amsgrad: step must be >= 1");
  if (n == 0) return 0;
  const double bc1 = 1.0 - pow((double)beta1, (double)step);
  const double bc2 = 1.0 - pow((double)beta2, (double)step);
  const long long threads = (n + 3) / 4;
  const int grid = (int)((threads + 255) / 256);
  adam_amsgrad_kernel<<<grid, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      p, g, m, v, vmax, reinterpret_cast<__nv_bfloat16*>(shadow_bf16), n, lr, beta1, beta2, eps, (float)bc1,
      (float)(1.0 / sqrt(bc2)), grad_scale, nullptr);
  TNR_LAUNCH_CHECK();
  return 0;
}

// step counter on the device: ++step, then the two bias corrections (double precision, one thread)
__global__ void adam_step_prep_kernel(int* __restrict__ step_dev, float* __restrict__ bc, float b1, float b2) {
  const int step = ++(*step_dev);
  bc[0] = (float)(1.0 - pow((double)b1, (double)step));
  bc[1] = (float)(1.0 / sqrt(1.0 - pow((double)b2, (double)step)));
}

TNR_API int tnr_adam_amsgrad_devstep(float* p, const float* g, float* m, float* v, float* vmax, void* shadow_bf16,
                                     long long n, float lr, float beta1, float beta2, float eps, int* step_dev,
                                     float* bc_ws, float grad_scale, int advance, void* stream) {
  TNR_REQUIRE(step_dev != nullptr && bc_ws != nullptr, "tnr_adam_amsgrad_devstep: step_dev (int32) and bc_ws (2 floats) are required");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (advance) {
    adam_step_prep_kernel<<<1, 1, 0, st>>>(step_dev, bc_ws, beta1, beta2);
    TNR_LAUNCH_CHECK();
  }
  if (n == 0) return 0;
  const long long threads = (n + 3) / 4;
  const int grid = (int)((threads + 255) / 256);
  adam_amsgrad_kernel<<<grid, 256, 0, st>>>(p, g, m, v, vmax, reinterpret_cast<__nv_bfloat16*>(shadow_bf16), n, lr, beta1,
                                            beta2, eps, 1.0f, 1.0f, grad_scale, bc_ws);
  TNR_LAUNCH_CHECK();
  return 0;
}

TNR_API int tnr_cast_f32_bf16(const float* x, void* y_bf16, long long n, void* stream) {
  if (n == 0) return 0;
  const long long threads = (n + 3) / 4;
  cast_f32_bf16_kernel<<<(int)((threads + 255) / 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      x, reinterpret_cast<__nv_bfloat16*>(y_bf16), n);
  TNR_LAUNCH_CHECK();
  return 0;
}

TNR_API int tnr_gather_rows_i32_i64(const int32_t* table, long long n_rows_table, const int32_t* idx, long long n, int W,
                                    int64_t* out, void* stream) {
  if (n == 0) return 0;
  gather_rows_i32_i64_kernel<<<(int)((n + 8 * GI_ROWS - 1) / (8 * GI_ROWS)), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      table, n_rows_table, idx, n, W, out);
  TNR_LAUNCH_CHECK();
  return 0;
}

TNR_API int tnr_gather_rows_f32(const float* table, long long n_rows_table, const int32_t* idx, long long n, int D,
                                float* out, long long out_ld, void* stream) {
  TNR_REQUIRE(D % 4 == 0 && out_ld % 4 == 0, "tnr_gather_rows_f32: D and out_ld must be multiples of 4");
  if (n == 0) return 0;
  gather_rows_f32_kernel<<<(int)((n + 7) / 8), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(table, n_rows_table, idx,
                                                                                                  n, D, out, out_ld);
  TNR_LAUNCH_CHECK();
  return 0;
}

TNR_API int tnr_train_batch_gather(const int32_t* news, long long n_rows, int W, const float* const* teacher_tables,
                                   float* const* teacher_out, int M, int D, long long out_ld, const int32_t* hist_idx,
                                   long long n_hist, const int32_t* cand_idx, long long n_cand, long long* tokens_out,
                                   void* stream) {
  TNR_REQUIRE(M >= 0 && M <= TB_MAX_TEACHERS, "tnr_train_batch_gather: at most %d teacher tables (got %d)", TB_MAX_TEACHERS, M);
  TNR_REQUIRE(M == 0 || (D % 4 == 0 && out_ld % 4 == 0 && teacher_tables != nullptr && teacher_out != nullptr),
              "tnr_train_batch_gather: D and out_ld must be multiples of 4");
  TNR_REQUIRE(news != nullptr && tokens_out != nullptr && n_rows >= 1 && W >= 1, "tnr_train_batch_gather: token table / output required");
  if (n_hist + n_cand == 0) return 0;
  TrainBatchGather g;
  g.news = news; g.n_rows = n_rows; g.W = W; g.M = M; g.D = D; g.out_ld = out_ld;
  for (int i = 0; i < TB_MAX_TEACHERS; ++i) {
    g.teacher[i] = i < M ? teacher_tables[i] : nullptr;
    g.teacher_out[i] = i < M ? teacher_out[i] : nullptr;
  }
  g.hist_idx = hist_idx; g.cand_idx = cand_idx; g.n_hist = n_hist; g.n_cand = n_cand; g.tokens_out = tokens_out;
  const dim3 grid((unsigned)((n_hist + n_cand + 7) / 8), (unsigned)(1 + M));
  train_batch_gather_kernel<<<grid, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(g);
  TNR_LAUNCH_CHECK();
  return 0;
}

TNR_API int tnr_doc_sim(const float* table, long long n_rows, const int32_t* pairs, long long n_pairs, int D,
                        double* sum_out, void* stream) {
  TNR_REQUIRE(D % 4 == 0 && D > 0, "tnr_doc_sim: D=%d must be a positive multiple of 4", D);
  TNR_REQUIRE(sum_out != nullptr, "tnr_doc_sim: sum_out (one double, caller-initialised) is required");
  if (n_pairs == 0) return 0;
  doc_sim_kernel<<<(int)((n_pairs + 7) / 8), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(table, n_rows, pairs, n_pairs, D,
                                                                                             sum_out);
  TNR_LAUNCH_CHECK();
  return 0;
}

template <int VPL>
static void eval_score_launch(int grid, cudaStream_t st, const float* table, long long n_rows, const float* user,
                              const long long* ptr, const int32_t* cand, long long n_imp, long long nnz, float* score) {
  eval_score_kernel<VPL><<<grid, ES_WARPS * 32, 0, st>>>(table, n_rows, user, ptr, cand, n_imp, nnz, score);
}

int tnr::eval_scores(const char* what, const float* table, long long n_rows, const float* user, const long long* ptr,
                const int32_t* cand, long long n_imp, long long nnz, int D, float* scores, cudaStream_t st) {
  if (nnz == 0) return 0;
  const long long items = (nnz + ES_CPW - 1) / ES_CPW;
  long long blocks = (items + ES_WARPS - 1) / ES_WARPS;
  const long long cap_blocks = (long long)num_sms() * 8;
  const int grid = (int)(blocks < cap_blocks ? blocks : cap_blocks);
  switch (D / 32) {
    case 1: eval_score_launch<1>(grid, st, table, n_rows, user, ptr, cand, n_imp, nnz, scores); break;
    case 2: eval_score_launch<2>(grid, st, table, n_rows, user, ptr, cand, n_imp, nnz, scores); break;
    case 4: eval_score_launch<4>(grid, st, table, n_rows, user, ptr, cand, n_imp, nnz, scores); break;
    case 8: eval_score_launch<8>(grid, st, table, n_rows, user, ptr, cand, n_imp, nnz, scores); break;
    case 16: eval_score_launch<16>(grid, st, table, n_rows, user, ptr, cand, n_imp, nnz, scores); break;
    default:
      set_error("%s: D=%d not instantiated (32, 64, 128, 256, 512)", what, D);
      return 1;
  }
  TNR_LAUNCH_CHECK();
  return 0;
}

TNR_API int tnr_eval_metrics(const float* table, long long n_rows, const float* user, const long long* ptr,
                             const int32_t* cand, const int8_t* label, long long n_imp, long long nnz, int D, int max_c,
                             double* per_imp, double* sums, float* scores, void* stream) {
  TNR_REQUIRE(D % 32 == 0 && D >= 32 && D <= 512, "tnr_eval_metrics: D=%d must be a multiple of 32 in 32..512", D);
  TNR_REQUIRE(scores != nullptr || nnz == 0, "tnr_eval_metrics: scores fp32 [nnz] is required (output and workspace)");
  TNR_REQUIRE(n_rows >= 1, "tnr_eval_metrics: empty table");
  if (n_imp == 0) return 0;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (eval_scores("tnr_eval_metrics", table, n_rows, user, ptr, cand, n_imp, nnz, D, scores, st)) return 1;
  // rank kernel: a warp per impression holds its scores, positive list and labels in shared memory (9 bytes per candidate)
  const int cap = ((max_c > 1 ? max_c : 1) + 15) / 16 * 16;
  int wpb = ER_WARPS;
  while (wpb > 1 && (size_t)wpb * cap * 9 > 160 * 1024) wpb >>= 1;
  const size_t smem = (size_t)wpb * cap * 9;
  TNR_REQUIRE(smem <= 200 * 1024, "tnr_eval_metrics: max candidates %d too large", max_c);
  if (smem > 48 * 1024) TNR_SET_SMEM(eval_rank_kernel, smem);
  eval_rank_kernel<<<(unsigned)((n_imp + wpb - 1) / wpb), wpb * 32, smem, st>>>(scores, ptr, label, n_imp, cap, per_imp);
  TNR_LAUNCH_CHECK();
  if (sums != nullptr) {
    int grid = (int)((n_imp + 255) / 256);
    if (grid > 592) grid = 592;
    eval_reduce_kernel<<<grid, 256, 0, st>>>(per_imp, n_imp, sums);
    TNR_LAUNCH_CHECK();
  }
  return 0;
}
