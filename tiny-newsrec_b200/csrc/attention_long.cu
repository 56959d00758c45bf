// Self-attention with relative-position bias for 32 < L <= 512 (body / abstract text, table build of
// title+abstract+body rows), head dim 64: forward (below) and backward (second half of the file).
//   P = softmax(Q K^T / 8 + (1 - mask) * -10000 + relbias[h][j - i]);  ctx = dropout(P) V
// Reference: Tiny-NewsRec/tnlrv3/modeling.py:205-231, mask :446-454, rel-pos bias :458-463.
//
// One block (4 warps, 4 blocks per SM) per (news, head, 64-query block); each warp owns 16 query rows.  K / V
// are streamed through a double-buffered shared-memory stage in 64-key chunks (cp.async, the next chunk in
// flight while the current one is used), the two contractions run on ldmatrix + mma.sync
// m16n8k16 (bf16 in, fp32 accumulate) with the usual online softmax (running max / sum per row, the output
// accumulator rescaled when the max moves), so nothing of size L x L is ever materialised.  The bias is a
// function of j - i only: the per-head [2L-1] vector and the additive key mask live in shared memory.
// Arithmetic intensity is 4 L E / (8 E) = L / 2 FLOP/B: HBM-bound below L ~ 400 on B200.
#include "common.cuh"
#include "mma_sync.cuh"

namespace tnr {

constexpr int LDH = 64;            // head dim
constexpr int LQB = 64;            // query rows per block
constexpr int LKB = 64;            // keys per chunk
constexpr int LTS = 72;            // smem row stride (bf16): 144 B, ldmatrix conflict-free
constexpr int LONG_LMAX = 512;

// rows [r0, r0 + 64) x 64 bf16 of a [L, ld] matrix -> padded smem tile; rows >= L zero-filled. 128 threads.
__device__ __forceinline__ void long_load_tile(__nv_bfloat16* s, const __nv_bfloat16* g, int r0, int L, int ld, int tid) {
#pragma unroll
  for (int it = 0; it < 4; ++it) {
    const int idx = tid + 128 * it, r = idx >> 3, c = idx & 7;
    if (r0 + r < L) cp_async16(smem_addr(s + r * LTS + c * 8), g + (size_t)(r0 + r) * ld + c * 8);
    else *reinterpret_cast<uint4*>(s + r * LTS + c * 8) = make_uint4(0, 0, 0, 0);
  }
}

constexpr float LOG2E = 1.4426950408889634f;

__device__ __forceinline__ void cp_async_commit_group() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait_group() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

__global__ void __launch_bounds__(128, 4)
attn_long_fwd_kernel(const __nv_bfloat16* __restrict__ qkv, const int64_t* __restrict__ mask, int mask_ld,
                     const float* __restrict__ relbias, __nv_bfloat16* __restrict__ ctx, int n_news, int L, int A, int E,
                     int q_blocks, const tnr_dropout drop) {
  extern __shared__ __align__(16) uint8_t smem[];
  __nv_bfloat16* sQ = reinterpret_cast<__nv_bfloat16*>(smem);
  __nv_bfloat16* sKV = sQ + LQB * LTS;                           // [2 buffers][K tile | V tile]
  const int k_chunks = (L + LKB - 1) / LKB;
  float* s_madd = reinterpret_cast<float*>(sKV + 4 * LKB * LTS);  // [k_chunks * 64], pre-multiplied by log2(e)
  float* s_rel = s_madd + k_chunks * LKB;                         // [2L - 1 (+ 64 zeros)], pre-multiplied by log2(e)
  __shared__ int s_live[LONG_LMAX / LKB];                         // chunk holds at least one unmasked key
  __shared__ int s_any;
  const int tid = threadIdx.x, warp = uniform_warp_id(), lane = tid & 31;
  const int g = lane >> 2, t = lane & 3;
  const long long item = blockIdx.x / q_blocks;
  const int qb = blockIdx.x % q_blocks;
  const int n = (int)(item / A), h = (int)(item % A);
  const int q0 = qb * LQB;
  const int ld = 3 * E;
  const __nv_bfloat16* base = qkv + (size_t)n * L * ld + h * LDH;
  const DropCfg dc = load_drop(drop);

  long_load_tile(sQ, base, q0, L, ld, tid);
  long_load_tile(sKV, base + E, 0, L, ld, tid);
  long_load_tile(sKV + LKB * LTS, base + 2 * E, 0, L, ld, tid);
  cp_async_commit_group();
  if (tid < LONG_LMAX / LKB) s_live[tid] = 0;
  if (tid == 0) s_any = 0;
  __syncthreads();
  for (int j = tid; j < k_chunks * LKB; j += 128) {
    float v = -INFINITY;
    if (j < L) {
      const bool keep = mask[(size_t)n * mask_ld + j] != 0;
      v = keep ? 0.f : -10000.0f * LOG2E;
      if (keep) { s_live[j / LKB] = 1; s_any = 1; }             // benign race: every writer stores 1
    }
    s_madd[j] = v;
  }
  for (int d = tid; d < 2 * L - 1 + LKB; d += 128)              // zero tail: keys j >= L index past the vector
    s_rel[d] = d < 2 * L - 1 ? relbias[(size_t)h * (2 * L - 1) + d] * LOG2E : 0.f;
  cp_async_wait_group<0>();
  __syncthreads();

  // Q fragments of this warp's 16 rows stay in registers for the whole key loop
  uint32_t qa[4][4];
#pragma unroll
  for (int ks = 0; ks < 4; ++ks)
    ldsm_x4(smem_addr(sQ + (warp * 16 + (lane & 7) + ((lane >> 3) & 1) * 8) * LTS + ks * 16 + (lane >> 4) * 8), qa[ks]);

  float o[8][4];
#pragma unroll
  for (int nt = 0; nt < 8; ++nt)
#pragma unroll
    for (int c = 0; c < 4; ++c) o[nt][c] = 0.f;
  float m_run[2] = {-INFINITY, -INFINITY}, l_run[2] = {0.f, 0.f};
  const int i0 = q0 + warp * 16 + g;                 // this thread's rows: i0 and i0 + 8
  const bool warp_live = q0 + warp * 16 < L;         // warp-uniform: rows beyond L produce nothing
  // A chunk whose keys are all masked (additive -10000) contributes exactly 0 to every row as soon as the
  // news has one unmasked key anywhere (exp underflows in fp32), so it is skipped; an all-pad news keeps
  // every chunk (uniform shift, the reference's result).
  const bool any_key = s_any != 0;

  for (int kc = 0; kc < k_chunks; ++kc) {
    const int c0 = kc * LKB;
    const __nv_bfloat16* sK = sKV + (kc & 1) * 2 * LKB * LTS;
    const __nv_bfloat16* sV = sK + LKB * LTS;
    if (kc + 1 < k_chunks) {                         // prefetch the next chunk into the other buffer
      __nv_bfloat16* nK = sKV + ((kc + 1) & 1) * 2 * LKB * LTS;
      long_load_tile(nK, base + E, c0 + LKB, L, ld, tid);
      long_load_tile(nK + LKB * LTS, base + 2 * E, c0 + LKB, L, ld, tid);
      cp_async_commit_group();
      cp_async_wait_group<1>();
    } else {
      cp_async_wait_group<0>();
    }
    __syncthreads();                                 // chunk kc visible to all warps
    if (warp_live && (s_live[kc] || !any_key)) {
      float s[8][4];
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
        for (int c = 0; c < 4; ++c) s[nt][c] = 0.f;
        uint32_t kb[2][4];
#pragma unroll
        for (int half = 0; half < 2; ++half)
          ldsm_x4(smem_addr(sK + (nt * 8 + (lane & 7)) * LTS + half * 32 + (lane >> 3) * 8), kb[half]);
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) mma_bf16(s[nt], qa[ks], kb[ks >> 1][(ks & 1) * 2], kb[ks >> 1][(ks & 1) * 2 + 1]);
      }
      // scores (in log2 units) -> probabilities of this chunk under the running maximum.  Keys j >= L carry
      // s_madd = -inf (no bound check).  The additive terms of this thread's 16 columns are fetched once: the
      // key mask is shared by both rows, and row i0 + 8 sees the rel-pos values of row i0 eight keys earlier.
      {
        const int ib = min(i0, L - 1);
        const float* relp = s_rel + (L - 1 - ib) + c0 + 2 * t;         // rel of (row i0, key c0 + 2t + ...)
        float rel[9][2];
#pragma unroll
        for (int nt = 0; nt < 9; ++nt) {
          const int off = (nt - 1) * 8;                                   // nt = 0: the eight keys before the chunk
          const bool ok = (L - 1 - ib) + c0 + 2 * t + off >= 0;
          rel[nt][0] = ok ? relp[off] : 0.f;
          rel[nt][1] = ok ? relp[off + 1] : 0.f;
        }
        const bool row1_clamped = i0 + 8 > L - 1;                        // tail rows reuse row L-1 (never stored)
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
          const float2 md = *reinterpret_cast<const float2*>(s_madd + c0 + nt * 8 + 2 * t);
          const f32x2 mdp = pk2(md.x, md.y);
          const f32x2 a0 = add2(mdp, pk2(rel[nt + 1][0], rel[nt + 1][1]));
          const f32x2 a1 = add2(mdp, row1_clamped ? pk2(rel[nt + 1][0], rel[nt + 1][1]) : pk2(rel[nt][0], rel[nt][1]));
          const f32x2 sc = pk2(0.125f * LOG2E, 0.125f * LOG2E);
          upk2(fma2(pk2(s[nt][0], s[nt][1]), sc, a0), s[nt][0], s[nt][1]);
          upk2(fma2(pk2(s[nt][2], s[nt][3]), sc, a1), s[nt][2], s[nt][3]);
        }
      }
#pragma unroll
      for (int hi = 0; hi < 2; ++hi) {
        float mx = -INFINITY;
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) mx = fmaxf(mx, fmaxf(s[nt][hi * 2], s[nt][hi * 2 + 1]));
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
        const float m_new = fmaxf(m_run[hi], mx);    // finite: a processed chunk holds at least one key j < L
        const float corr = ex2_approx(m_run[hi] - m_new);   // 2^-inf = 0 on the first chunk
        const f32x2 mneg = pk2(-m_new, -m_new);
        f32x2 sum2 = pk2(0.f, 0.f);
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
          float x0, x1;
          upk2(add2(pk2(s[nt][hi * 2], s[nt][hi * 2 + 1]), mneg), x0, x1);
          s[nt][hi * 2] = ex2_approx(x0);
          s[nt][hi * 2 + 1] = ex2_approx(x1);
          sum2 = add2(sum2, pk2(s[nt][hi * 2], s[nt][hi * 2 + 1]));
        }
        float sa, sb;
        upk2(sum2, sa, sb);
        float sum = sa + sb;
        sum += __shfl_xor_sync(0xffffffffu, sum, 1);
        sum += __shfl_xor_sync(0xffffffffu, sum, 2);
        l_run[hi] = l_run[hi] * corr + sum;
        m_run[hi] = m_new;
        const f32x2 c2 = pk2(corr, corr);
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) upk2(mul2(pk2(o[nt][hi * 2], o[nt][hi * 2 + 1]), c2), o[nt][hi * 2], o[nt][hi * 2 + 1]);
      }
      if (dc.thr16 != 0) {
        // dropout on the (unnormalised) probabilities; the 1/(1-p) scale commutes with the final 1/l.
        // Philox group of (item, i, chunk kc, quad lane t, half of the chunk): 8 elements, bit (nt & 3) * 2 + e.
#pragma unroll
        for (int hi = 0; hi < 2; ++hi) {
          const uint64_t row = (uint64_t)item * (uint64_t)L + (uint64_t)min(i0 + hi * 8, L - 1);
#pragma unroll
          for (int hf = 0; hf < 2; ++hf) {
            const uint32_t keep = dropout_keep8(dc, ((row * (uint64_t)k_chunks + (uint64_t)kc) * 4 + (uint64_t)t) * 2 + hf);
#pragma unroll
            for (int q = 0; q < 4; ++q)
#pragma unroll
              for (int e = 0; e < 2; ++e)
                s[hf * 4 + q][hi * 2 + e] = ((keep >> (q * 2 + e)) & 1u) ? s[hf * 4 + q][hi * 2 + e] * dc.scale : 0.f;
          }
        }
      }
      // P (16 x 64, C layout) -> A fragments; O += P V
      uint32_t pa[4][4];
#pragma unroll
      for (int ks = 0; ks < 4; ++ks) {
        pa[ks][0] = pack_bf16(s[2 * ks][0], s[2 * ks][1]);
        pa[ks][1] = pack_bf16(s[2 * ks][2], s[2 * ks][3]);
        pa[ks][2] = pack_bf16(s[2 * ks + 1][0], s[2 * ks + 1][1]);
        pa[ks][3] = pack_bf16(s[2 * ks + 1][2], s[2 * ks + 1][3]);
      }
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
        for (int kh = 0; kh < 2; ++kh) {             // keys 0-31, 32-63 of the chunk
          uint32_t vb[4];
          ldsm_x4_t(smem_addr(sV + (kh * 32 + lane) * LTS + nt * 8), vb);
          mma_bf16(o[nt], pa[kh * 2], vb[0], vb[1]);
          mma_bf16(o[nt], pa[kh * 2 + 1], vb[2], vb[3]);
        }
      }
    }
    __syncthreads();                                 // chunk kc consumed: its buffer may be refilled
  }
  if (!warp_live) return;
  // normalise, stage this warp's 16 x 64 rows in its own (already consumed) part of sQ, store full 128 B rows
  const float inv0 = 1.0f / l_run[0], inv1 = 1.0f / l_run[1];
  __nv_bfloat16* sO = sQ + warp * 16 * LTS;
#pragma unroll
  for (int nt = 0; nt < 8; ++nt) {
    *reinterpret_cast<uint32_t*>(sO + g * LTS + nt * 8 + 2 * t) = pack_bf16(o[nt][0] * inv0, o[nt][1] * inv0);
    *reinterpret_cast<uint32_t*>(sO + (g + 8) * LTS + nt * 8 + 2 * t) = pack_bf16(o[nt][2] * inv1, o[nt][3] * inv1);
  }
  __syncwarp();
  __nv_bfloat16* obase = ctx + (size_t)n * L * E + h * LDH;
#pragma unroll
  for (int it = 0; it < 4; ++it) {
    const int idx = lane + 32 * it, r = idx >> 3, c = idx & 7;
    const int row = q0 + warp * 16 + r;
    if (row < L) *reinterpret_cast<uint4*>(obase + (size_t)row * E + c * 8) = *reinterpret_cast<const uint4*>(sO + r * LTS + c * 8);
  }
}

// ---------------------------------------------------------------------------------------------------
// Backward for 32 < L <= 512, two kernels, no atomics on the gradients (deterministic):
//   dq kernel : block per (news, head, 64-query block), K / V streamed TWICE.  Sweep 1 recomputes the scores and
//               dP = dO V^T and keeps, online (as the forward keeps m and l), the row maximum, the row sum and
//               delta_i = sum_j P_ij dP_ij -- so neither the forward's statistics nor its output are needed.
//               Sweep 2 forms dS = P o (dP - delta) / 8 chunk by chunk and accumulates dQ = dS K.  It also
//               writes lse_i (log2 units) and delta_i for the second kernel.
//   dkv kernel: block per (news, head, 64-key block), K / V tiles resident, Q / dO streamed in 64-query chunks.
//               Phase 1 (warp = 16 queries, the forward's layout, so the dropout bits are the forward's):
//               P~ = dropout(P) and dS into shared memory; phase 2 (warp = 16 keys): dV += P~^T dO,
//               dK += dS^T Q with the transposed fragments read by ldmatrix.trans.
// dP_eff = dP o keep / (1 - p) throughout (gradient w.r.t. the pre-dropout probability).
// Reference: the autograd backward of tnlrv3/modeling.py:205-231.
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ void lb_load_a(uint32_t (&a)[4][4], const __nv_bfloat16* sA, int row0, int lane) {
#pragma unroll
  for (int ks = 0; ks < 4; ++ks)
    ldsm_x4(smem_addr(sA + (row0 + (lane & 7) + ((lane >> 3) & 1) * 8) * LTS + ks * 16 + (lane >> 4) * 8), a[ks]);
}
// A fragments of T^T for the 16 columns [m0, m0 + 16) of a 64 x 64 tile T (rows = the contraction index)
__device__ __forceinline__ void lb_load_aT(uint32_t (&a)[4][4], const __nv_bfloat16* sT, int m0, int lane) {
  const int mi = lane >> 3;
#pragma unroll
  for (int ks = 0; ks < 4; ++ks)
    ldsm_x4_t(smem_addr(sT + (ks * 16 + (lane & 7) + (mi >> 1) * 8) * LTS + m0 + (mi & 1) * 8), a[ks]);
}
// s[nt] = A (16 x 64) . B^T, B tile = 64 rows (n) x 64 (k)
__device__ __forceinline__ void lb_mma_abT(float (&s)[8][4], const uint32_t (&a)[4][4], const __nv_bfloat16* sB, int lane) {
#pragma unroll
  for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
    for (int c = 0; c < 4; ++c) s[nt][c] = 0.f;
    uint32_t kb[2][4];
#pragma unroll
    for (int half = 0; half < 2; ++half)
      ldsm_x4(smem_addr(sB + (nt * 8 + (lane & 7)) * LTS + half * 32 + (lane >> 3) * 8), kb[half]);
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) mma_bf16(s[nt], a[ks], kb[ks >> 1][(ks & 1) * 2], kb[ks >> 1][(ks & 1) * 2 + 1]);
  }
}
// o[nt] += P (16 x 64, A fragments) . B, B tile = 64 rows (k) x 64 (n)
__device__ __forceinline__ void lb_mma_pb(float (&o)[8][4], const uint32_t (&pa)[4][4], const __nv_bfloat16* sB, int lane) {
#pragma unroll
  for (int nt = 0; nt < 8; ++nt)
#pragma unroll
    for (int kh = 0; kh < 2; ++kh) {
      uint32_t vb[4];
      ldsm_x4_t(smem_addr(sB + (kh * 32 + lane) * LTS + nt * 8), vb);
      mma_bf16(o[nt], pa[kh * 2], vb[0], vb[1]);
      mma_bf16(o[nt], pa[kh * 2 + 1], vb[2], vb[3]);
    }
}
__device__ __forceinline__ void lb_c_to_a(uint32_t (&pa)[4][4], const float (&s)[8][4]) {
#pragma unroll
  for (int ks = 0; ks < 4; ++ks) {
    pa[ks][0] = pack_bf16(s[2 * ks][0], s[2 * ks][1]);
    pa[ks][1] = pack_bf16(s[2 * ks][2], s[2 * ks][3]);
    pa[ks][2] = pack_bf16(s[2 * ks + 1][0], s[2 * ks + 1][1]);
    pa[ks][3] = pack_bf16(s[2 * ks + 1][2], s[2 * ks + 1][3]);
  }
}
// raw QK^T accumulators -> scores in log2 units with the key mask and the rel-pos bias added (the forward's code):
// rows i0 (c = 0, 1) and i0 + 8 (c = 2, 3), keys c0 + nt * 8 + 2 t + {0, 1}.  s_madd is indexed from key c0.
__device__ __forceinline__ void lb_add_bias(float (&s)[8][4], const float* s_madd_c0, const float* s_rel, int i0, int c0, int L,
                                            int t) {
  const int ib = min(i0, L - 1);
  const float* relp = s_rel + (L - 1 - ib) + c0 + 2 * t;
  float rel[9][2];
#pragma unroll
  for (int nt = 0; nt < 9; ++nt) {
    const int off = (nt - 1) * 8;
    const bool ok = (L - 1 - ib) + c0 + 2 * t + off >= 0;
    rel[nt][0] = ok ? relp[off] : 0.f;
    rel[nt][1] = ok ? relp[off + 1] : 0.f;
  }
  const bool row1_clamped = i0 + 8 > L - 1;
#pragma unroll
  for (int nt = 0; nt < 8; ++nt) {
    const float2 md = *reinterpret_cast<const float2*>(s_madd_c0 + nt * 8 + 2 * t);
    const float sc = 0.125f * LOG2E;
    s[nt][0] = fmaf(s[nt][0], sc, md.x + rel[nt + 1][0]);
    s[nt][1] = fmaf(s[nt][1], sc, md.y + rel[nt + 1][1]);
    s[nt][2] = fmaf(s[nt][2], sc, md.x + (row1_clamped ? rel[nt + 1][0] : rel[nt][0]));
    s[nt][3] = fmaf(s[nt][3], sc, md.y + (row1_clamped ? rel[nt + 1][1] : rel[nt][1]));
  }
}
// keep * scale factors of this thread's 2 x 16 elements of (rows i0 / i0 + 8, key chunk kc): the forward's Philox groups
__device__ __forceinline__ void lb_keep(float (&kf)[8][4], const DropCfg& dc, long long item, int L, int i0, int k_chunks, int kc,
                                        int t) {
#pragma unroll
  for (int hi = 0; hi < 2; ++hi) {
    const uint64_t row = (uint64_t)item * (uint64_t)L + (uint64_t)min(i0 + hi * 8, L - 1);
#pragma unroll
    for (int hf = 0; hf < 2; ++hf) {
      const uint32_t keep = dropout_keep8(dc, ((row * (uint64_t)k_chunks + (uint64_t)kc) * 4 + (uint64_t)t) * 2 + hf);
#pragma unroll
      for (int q = 0; q < 4; ++q)
#pragma unroll
        for (int e = 0; e < 2; ++e) kf[hf * 4 + q][hi * 2 + e] = ((keep >> (q * 2 + e)) & 1u) ? dc.scale : 0.f;
    }
  }
}

// the same, multiplied into dp in place (dP_eff)
__device__ __forceinline__ void lb_apply_keep(float (&dp)[8][4], const DropCfg& dc, long long item, int L, int i0, int k_chunks,
                                              int kc, int t) {
#pragma unroll
  for (int hi = 0; hi < 2; ++hi) {
    const uint64_t row = (uint64_t)item * (uint64_t)L + (uint64_t)min(i0 + hi * 8, L - 1);
#pragma unroll
    for (int hf = 0; hf < 2; ++hf) {
      const uint32_t keep = dropout_keep8(dc, ((row * (uint64_t)k_chunks + (uint64_t)kc) * 4 + (uint64_t)t) * 2 + hf);
#pragma unroll
      for (int q = 0; q < 4; ++q)
#pragma unroll
        for (int e = 0; e < 2; ++e) dp[hf * 4 + q][hi * 2 + e] *= ((keep >> (q * 2 + e)) & 1u) ? dc.scale : 0.f;
    }
  }
}

// DREL: also the rel-pos bias gradient.  Sweep 2 parks each chunk's dS (fp32, before the bf16 staging) in a per-warp
// tile and adds its diagonals, in chunk order, to a per-warp [2L-1] vector of diagonal sums; after the sweep the four
// vectors are added in warp order and folded into buckets -> part[blockIdx.x * nb + b] (relgrad_reduce_kernel).
constexpr int DT_LD = 65;          // row stride (floats) of the per-warp 16 x 64 dS tile
template <bool DREL>
__device__ __forceinline__ void attn_long_bwd_dq_body(const __nv_bfloat16* __restrict__ qkv, const int64_t* __restrict__ mask,
                                                      int mask_ld, const float* __restrict__ relbias,
                                                      const __nv_bfloat16* __restrict__ dctx, __nv_bfloat16* __restrict__ dqkv,
                                                      float* __restrict__ dbias, float* __restrict__ ws_lse,
                                                      float* __restrict__ ws_delta, int n_news, int L, int A, int E, int q_blocks,
                                                      const tnr_dropout& drop, const int* __restrict__ bucket, int nb,
                                                      float* __restrict__ part) {
  extern __shared__ __align__(16) uint8_t smem[];
  __nv_bfloat16* sQ = reinterpret_cast<__nv_bfloat16*>(smem);
  __nv_bfloat16* sdO = sQ + LQB * LTS;
  __nv_bfloat16* sKV = sdO + LQB * LTS;                           // [2 buffers][K tile | V tile]
  const int k_chunks = (L + LKB - 1) / LKB;
  float* s_madd = reinterpret_cast<float*>(sKV + 4 * LKB * LTS);  // [k_chunks * 64]
  float* s_rel = s_madd + k_chunks * LKB;                         // [2L - 1 (+ 64 zeros)]
  __shared__ int s_live[LONG_LMAX / LKB];
  __shared__ int s_any;
  const int tid = threadIdx.x, warp = uniform_warp_id(), lane = tid & 31;
  const int g = lane >> 2, t = lane & 3;
  const long long item = blockIdx.x / q_blocks;
  const int qb = blockIdx.x % q_blocks;
  const int n = (int)(item / A), h = (int)(item % A);
  const int q0 = qb * LQB;
  const int ld = 3 * E;
  const __nv_bfloat16* base = qkv + (size_t)n * L * ld + h * LDH;
  const DropCfg dc = load_drop(drop);

  long_load_tile(sQ, base, q0, L, ld, tid);
  long_load_tile(sdO, dctx + (size_t)n * L * E + h * LDH, q0, L, E, tid);
  long_load_tile(sKV, base + E, 0, L, ld, tid);
  long_load_tile(sKV + LKB * LTS, base + 2 * E, 0, L, ld, tid);
  cp_async_commit_group();
  if (tid < LONG_LMAX / LKB) s_live[tid] = 0;
  if (tid == 0) s_any = 0;
  __syncthreads();
  for (int j = tid; j < k_chunks * LKB; j += 128) {
    float v = -INFINITY;
    if (j < L) {
      const bool keep = mask[(size_t)n * mask_ld + j] != 0;
      v = keep ? 0.f : -10000.0f * LOG2E;
      if (keep) { s_live[j / LKB] = 1; s_any = 1; }
    }
    s_madd[j] = v;
  }
  for (int d = tid; d < 2 * L - 1 + LKB; d += 128)
    s_rel[d] = d < 2 * L - 1 ? relbias[(size_t)h * (2 * L - 1) + d] * LOG2E : 0.f;
  float* s_dacc = s_rel + 2 * L - 1 + LKB;                        // DREL: [4 warps][2L] diagonal sums
  float* s_dt = s_dacc + 8 * L;                                   // DREL: [4 warps][16][DT_LD] dS tile
  if constexpr (DREL)
    for (int k = tid; k < 8 * L; k += 128) s_dacc[k] = 0.f;
  cp_async_wait_group<0>();
  __syncthreads();

  uint32_t qa[4][4], da[4][4];
  lb_load_a(qa, sQ, warp * 16, lane);
  lb_load_a(da, sdO, warp * 16, lane);
  const int i0 = q0 + warp * 16 + g;
  const bool warp_live = q0 + warp * 16 < L;
  const bool any_key = s_any != 0;
  float m_run[2] = {-INFINITY, -INFINITY}, l_run[2] = {0.f, 0.f}, d_run[2] = {0.f, 0.f};
  float lse[2] = {0.f, 0.f}, delta[2] = {0.f, 0.f};
  float dq[8][4];
#pragma unroll
  for (int nt = 0; nt < 8; ++nt)
#pragma unroll
    for (int c = 0; c < 4; ++c) dq[nt][c] = 0.f;

  for (int sweep = 0; sweep < 2; ++sweep) {
    for (int kc = 0; kc < k_chunks; ++kc) {
      const int c0 = kc * LKB;
      const int it = sweep * k_chunks + kc;          // the two sweeps share one double-buffered stream of 2 k_chunks items
      const __nv_bfloat16* sK = sKV + (it & 1) * 2 * LKB * LTS;
      const __nv_bfloat16* sV = sK + LKB * LTS;
      if (it + 1 < 2 * k_chunks) {                   // prefetch the next item (chunk 0 again after the first sweep)
        const int nc = kc + 1 < k_chunks ? kc + 1 : 0;
        __nv_bfloat16* nK = sKV + ((it + 1) & 1) * 2 * LKB * LTS;
        long_load_tile(nK, base + E, nc * LKB, L, ld, tid);
        long_load_tile(nK + LKB * LTS, base + 2 * E, nc * LKB, L, ld, tid);
        cp_async_commit_group();
        cp_async_wait_group<1>();
      } else {
        cp_async_wait_group<0>();
      }
      __syncthreads();
      if (warp_live && (s_live[kc] || !any_key)) {
        float s[8][4], dp[8][4];
        lb_mma_abT(s, qa, sK, lane);
        lb_add_bias(s, s_madd + c0, s_rel, i0, c0, L, t);
        lb_mma_abT(dp, da, sV, lane);
        if (dc.thr16 != 0) lb_apply_keep(dp, dc, item, L, i0, k_chunks, kc, t);
        if (sweep == 0) {
#pragma unroll
          for (int hi = 0; hi < 2; ++hi) {
            float mx = -INFINITY;
#pragma unroll
            for (int nt = 0; nt < 8; ++nt) mx = fmaxf(mx, fmaxf(s[nt][hi * 2], s[nt][hi * 2 + 1]));
            mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
            mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
            const float m_new = fmaxf(m_run[hi], mx);
            const float corr = ex2_approx(m_run[hi] - m_new);
            float sum = 0.f, dsum = 0.f;
#pragma unroll
            for (int nt = 0; nt < 8; ++nt)
#pragma unroll
              for (int e = 0; e < 2; ++e) {
                const float pv = ex2_approx(s[nt][hi * 2 + e] - m_new);
                sum += pv;
                dsum = fmaf(pv, dp[nt][hi * 2 + e], dsum);
              }
            l_run[hi] = l_run[hi] * corr + sum;           // per-thread partials: the quad is reduced after the sweep
            d_run[hi] = d_run[hi] * corr + dsum;
            m_run[hi] = m_new;
          }
        } else {
          float ds[8][4];
#pragma unroll
          for (int nt = 0; nt < 8; ++nt)
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              const int hi = c >> 1;
              const float pv = ex2_approx(s[nt][c] - lse[hi]);
              ds[nt][c] = pv * (dp[nt][c] - delta[hi]) * 0.125f;
            }
          uint32_t pa[4][4];
          lb_c_to_a(pa, ds);
          lb_mma_pb(dq, pa, sK, lane);
          if constexpr (DREL) {
            float* tw = s_dt + warp * 16 * DT_LD;
#pragma unroll
            for (int nt = 0; nt < 8; ++nt)
#pragma unroll
              for (int c = 0; c < 4; ++c) tw[(g + (c >> 1) * 8) * DT_LD + nt * 8 + 2 * t + (c & 1)] = ds[nt][c] * 8.0f;
            __syncwarp();
            // local diagonal dl = key - row in [-15, 63]: global j - i = c0 + dl - (q0 + 16 warp); rows / keys >= L are 0
            float* acc = s_dacc + warp * 2 * L;
            for (int dl = lane - 15; dl < LKB; dl += 32) {
              float sum = 0.f;
              for (int r = dl < 0 ? -dl : 0; r < 16 && r + dl < LKB; ++r) sum += tw[r * DT_LD + r + dl];
              const int k = c0 + dl - (q0 + warp * 16) + L - 1;
              if (k >= 0 && k < 2 * L - 1) acc[k] += sum;
            }
            __syncwarp();
          }
        }
      }
      __syncthreads();
    }
    if (sweep == 0) {
#pragma unroll
      for (int hi = 0; hi < 2; ++hi) {
        float l = l_run[hi], d = d_run[hi];
        l += __shfl_xor_sync(0xffffffffu, l, 1); l += __shfl_xor_sync(0xffffffffu, l, 2);
        d += __shfl_xor_sync(0xffffffffu, d, 1); d += __shfl_xor_sync(0xffffffffu, d, 2);
        lse[hi] = m_run[hi] + log2f(l);
        delta[hi] = d / l;
        const int i = i0 + hi * 8;
        if (warp_live && t == 0 && i < L) {
          ws_lse[(size_t)item * L + i] = lse[hi];
          ws_delta[(size_t)item * L + i] = delta[hi];
        }
      }
    }
  }
  if constexpr (DREL) {
    for (int k = tid; k < 2 * L - 1; k += 128)
      s_dacc[k] = ((s_dacc[k] + s_dacc[2 * L + k]) + s_dacc[4 * L + k]) + s_dacc[6 * L + k];
    __syncthreads();
    const int seg = (2 * L - 1 + 3) / 4;           // warp w folds diagonals [w seg, (w + 1) seg), lane = bucket
    const int k1 = min(2 * L - 1, (warp + 1) * seg);
    float a = 0.f;
    for (int k = warp * seg; k < k1; ++k)
      if (__ldg(bucket + k) == lane) a += s_dacc[k];
    s_dt[warp * 32 + lane] = a;
    __syncthreads();
    if (tid < nb) part[(size_t)blockIdx.x * nb + tid] = ((s_dt[tid] + s_dt[32 + tid]) + s_dt[64 + tid]) + s_dt[96 + tid];
  }
  if (!warp_live) return;
  __nv_bfloat16* sO = sQ + warp * 16 * LTS;       // this warp's (consumed) rows of sQ
#pragma unroll
  for (int nt = 0; nt < 8; ++nt) {
    *reinterpret_cast<uint32_t*>(sO + g * LTS + nt * 8 + 2 * t) = pack_bf16(dq[nt][0], dq[nt][1]);
    *reinterpret_cast<uint32_t*>(sO + (g + 8) * LTS + nt * 8 + 2 * t) = pack_bf16(dq[nt][2], dq[nt][3]);
  }
  __syncwarp();
  __nv_bfloat16* obase = dqkv + (size_t)n * L * ld + h * LDH;
#pragma unroll
  for (int it = 0; it < 4; ++it) {
    const int idx = lane + 32 * it, r = idx >> 3, c = idx & 7;
    const int row = q0 + warp * 16 + r;
    if (row < L) *reinterpret_cast<uint4*>(obase + (size_t)row * ld + c * 8) = *reinterpret_cast<const uint4*>(sO + r * LTS + c * 8);
  }
  if (dbias != nullptr) {                          // bq gradient: column sums of the bf16 rows just stored
    float a0 = 0.f, a1 = 0.f;
    for (int r = 0; r < 16 && q0 + warp * 16 + r < L; ++r) {
      const uint32_t u = *reinterpret_cast<const uint32_t*>(sO + r * LTS + 2 * lane);
      a0 += bf16_lo(u); a1 += bf16_hi(u);
    }
    atomicAdd(dbias + h * LDH + 2 * lane, a0);
    atomicAdd(dbias + h * LDH + 2 * lane + 1, a1);
  }
}

__global__ void __launch_bounds__(128, 2)
attn_long_bwd_dq_kernel(const __nv_bfloat16* __restrict__ qkv, const int64_t* __restrict__ mask, int mask_ld,
                        const float* __restrict__ relbias, const __nv_bfloat16* __restrict__ dctx,
                        __nv_bfloat16* __restrict__ dqkv, float* __restrict__ dbias, float* __restrict__ ws_lse,
                        float* __restrict__ ws_delta, int n_news, int L, int A, int E, int q_blocks, const tnr_dropout drop) {
  attn_long_bwd_dq_body<false>(qkv, mask, mask_ld, relbias, dctx, dqkv, dbias, ws_lse, ws_delta, n_news, L, A, E, q_blocks, drop,
                               nullptr, 0, nullptr);
}

__global__ void __launch_bounds__(128, 2)
attn_long_bwd_dq_drel_kernel(const __nv_bfloat16* __restrict__ qkv, const int64_t* __restrict__ mask, int mask_ld,
                             const float* __restrict__ relbias, const __nv_bfloat16* __restrict__ dctx,
                             __nv_bfloat16* __restrict__ dqkv, float* __restrict__ dbias, float* __restrict__ ws_lse,
                             float* __restrict__ ws_delta, int n_news, int L, int A, int E, int q_blocks, const tnr_dropout drop,
                             const int* __restrict__ bucket, int nb, float* __restrict__ part) {
  attn_long_bwd_dq_body<true>(qkv, mask, mask_ld, relbias, dctx, dqkv, dbias, ws_lse, ws_delta, n_news, L, A, E, q_blocks, drop,
                              bucket, nb, part);
}

__global__ void __launch_bounds__(128, 2)
attn_long_bwd_dkv_kernel(const __nv_bfloat16* __restrict__ qkv, const int64_t* __restrict__ mask, int mask_ld,
                         const float* __restrict__ relbias, const __nv_bfloat16* __restrict__ dctx,
                         __nv_bfloat16* __restrict__ dqkv, float* __restrict__ dbias, const float* __restrict__ ws_lse,
                         const float* __restrict__ ws_delta, int n_news, int L, int A, int E, int k_blocks,
                         const tnr_dropout drop) {
  extern __shared__ __align__(16) uint8_t smem[];
  __nv_bfloat16* sK = reinterpret_cast<__nv_bfloat16*>(smem);
  __nv_bfloat16* sV = sK + LKB * LTS;
  __nv_bfloat16* sQd = sV + LKB * LTS;                            // [2 buffers][Q tile | dO tile]
  __nv_bfloat16* sP = sQd + 4 * LQB * LTS;                        // [64 queries][64 keys]  dropout(P)
  __nv_bfloat16* sS = sP + LQB * LTS;                             // [64 queries][64 keys]  dS
  float* s_madd = reinterpret_cast<float*>(sS + LQB * LTS);       // [64] this key block
  float* s_rel = s_madd + LKB;                                    // [2L - 1 (+ 64 zeros)]
  __shared__ int s_any, s_live;
  const int tid = threadIdx.x, warp = uniform_warp_id(), lane = tid & 31;
  const int g = lane >> 2, t = lane & 3;
  const long long item = blockIdx.x / k_blocks;
  const int kb = blockIdx.x % k_blocks;
  const int n = (int)(item / A), h = (int)(item % A);
  const int c0 = kb * LKB;
  const int ld = 3 * E;
  const int q_chunks = (L + LQB - 1) / LQB;
  const __nv_bfloat16* base = qkv + (size_t)n * L * ld + h * LDH;
  const __nv_bfloat16* dobase = dctx + (size_t)n * L * E + h * LDH;
  const DropCfg dc = load_drop(drop);

  long_load_tile(sK, base + E, c0, L, ld, tid);
  long_load_tile(sV, base + 2 * E, c0, L, ld, tid);
  long_load_tile(sQd, base, 0, L, ld, tid);
  long_load_tile(sQd + LQB * LTS, dobase, 0, L, E, tid);
  cp_async_commit_group();
  if (tid == 0) { s_any = 0; s_live = 0; }
  __syncthreads();
  for (int j = tid; j < L; j += 128) {
    if (mask[(size_t)n * mask_ld + j] != 0) {
      s_any = 1;
      if (j >= c0 && j < c0 + LKB) s_live = 1;
    }
  }
  if (tid < LKB) {
    const int j = c0 + tid;
    s_madd[tid] = j < L ? (mask[(size_t)n * mask_ld + j] != 0 ? 0.f : -10000.0f * LOG2E) : -INFINITY;
  }
  for (int d = tid; d < 2 * L - 1 + LKB; d += 128)
    s_rel[d] = d < 2 * L - 1 ? relbias[(size_t)h * (2 * L - 1) + d] * LOG2E : 0.f;
  __syncthreads();
  const bool live = s_live != 0 || s_any == 0;     // a fully masked key block gets exactly zero probability

  float dk[8][4], dv[8][4];
#pragma unroll
  for (int nt = 0; nt < 8; ++nt)
#pragma unroll
    for (int c = 0; c < 4; ++c) { dk[nt][c] = 0.f; dv[nt][c] = 0.f; }

  for (int qc = 0; qc < q_chunks && live; ++qc) {
    const __nv_bfloat16* sQ = sQd + (qc & 1) * 2 * LQB * LTS;
    const __nv_bfloat16* sdO = sQ + LQB * LTS;
    if (qc + 1 < q_chunks) {
      __nv_bfloat16* nQ = sQd + ((qc + 1) & 1) * 2 * LQB * LTS;
      long_load_tile(nQ, base, (qc + 1) * LQB, L, ld, tid);
      long_load_tile(nQ + LQB * LTS, dobase, (qc + 1) * LQB, L, E, tid);
      cp_async_commit_group();
      cp_async_wait_group<1>();
    } else {
      cp_async_wait_group<0>();
    }
    __syncthreads();
    // ---- phase 1: this warp's 16 queries of the chunk against the 64 keys of the block
    {
      const int i0 = qc * LQB + warp * 16 + g;
      uint32_t qa[4][4], da[4][4];
      lb_load_a(qa, sQ, warp * 16, lane);
      lb_load_a(da, sdO, warp * 16, lane);
      float s[8][4], dp[8][4];
      lb_mma_abT(s, qa, sK, lane);
      lb_add_bias(s, s_madd, s_rel, i0, c0, L, t);
      lb_mma_abT(dp, da, sV, lane);
      float kf[8][4];
      if (dc.thr16 != 0) {
        lb_keep(kf, dc, item, L, i0, k_blocks, kb, t);
      } else {
#pragma unroll
        for (int nt = 0; nt < 8; ++nt)
#pragma unroll
          for (int c = 0; c < 4; ++c) kf[nt][c] = 1.f;
      }
      float lse[2], delta[2];
#pragma unroll
      for (int hi = 0; hi < 2; ++hi) {
        const int i = i0 + hi * 8;
        lse[hi] = i < L ? ws_lse[(size_t)item * L + i] : INFINITY;      // rows past L: probability 0
        delta[hi] = i < L ? ws_delta[(size_t)item * L + i] : 0.f;
      }
#pragma unroll
      for (int nt = 0; nt < 8; ++nt)
#pragma unroll
        for (int hi = 0; hi < 2; ++hi) {
          float pd[2], dsv[2];
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            const float pv = ex2_approx(s[nt][hi * 2 + e] - lse[hi]);
            pd[e] = pv * kf[nt][hi * 2 + e];
            dsv[e] = pv * (dp[nt][hi * 2 + e] * kf[nt][hi * 2 + e] - delta[hi]) * 0.125f;
          }
          const int r = warp * 16 + g + hi * 8;
          *reinterpret_cast<uint32_t*>(sP + r * LTS + nt * 8 + 2 * t) = pack_bf16(pd[0], pd[1]);
          *reinterpret_cast<uint32_t*>(sS + r * LTS + nt * 8 + 2 * t) = pack_bf16(dsv[0], dsv[1]);
        }
    }
    __syncthreads();
    // ---- phase 2: this warp's 16 keys: dV += P~^T dO, dK += dS^T Q
    {
      uint32_t pt[4][4];
      lb_load_aT(pt, sP, warp * 16, lane);
      lb_mma_pb(dv, pt, sdO, lane);
      lb_load_aT(pt, sS, warp * 16, lane);
      lb_mma_pb(dk, pt, sQ, lane);
    }
    __syncthreads();
  }
  if (!live) cp_async_wait_group<0>();
  __syncthreads();
  // dK -> sP, dV -> sS (this warp's 16 rows), then full 128-byte rows to global + bias column sums
  if (c0 + warp * 16 < L) {
    __nv_bfloat16* oK = sP + warp * 16 * LTS;
    __nv_bfloat16* oV = sS + warp * 16 * LTS;
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      *reinterpret_cast<uint32_t*>(oK + g * LTS + nt * 8 + 2 * t) = pack_bf16(dk[nt][0], dk[nt][1]);
      *reinterpret_cast<uint32_t*>(oK + (g + 8) * LTS + nt * 8 + 2 * t) = pack_bf16(dk[nt][2], dk[nt][3]);
      *reinterpret_cast<uint32_t*>(oV + g * LTS + nt * 8 + 2 * t) = pack_bf16(dv[nt][0], dv[nt][1]);
      *reinterpret_cast<uint32_t*>(oV + (g + 8) * LTS + nt * 8 + 2 * t) = pack_bf16(dv[nt][2], dv[nt][3]);
    }
    __syncwarp();
    __nv_bfloat16* obase = dqkv + (size_t)n * L * ld + h * LDH;
#pragma unroll
    for (int it = 0; it < 4; ++it) {
      const int idx = lane + 32 * it, r = idx >> 3, c = idx & 7;
      const int row = c0 + warp * 16 + r;
      if (row < L) {
        *reinterpret_cast<uint4*>(obase + (size_t)row * ld + E + c * 8) = *reinterpret_cast<const uint4*>(oK + r * LTS + c * 8);
        *reinterpret_cast<uint4*>(obase + (size_t)row * ld + 2 * E + c * 8) = *reinterpret_cast<const uint4*>(oV + r * LTS + c * 8);
      }
    }
    if (dbias != nullptr) {
      float k0 = 0.f, k1 = 0.f, v0 = 0.f, v1 = 0.f;
      for (int r = 0; r < 16 && c0 + warp * 16 + r < L; ++r) {
        const uint32_t uk = *reinterpret_cast<const uint32_t*>(oK + r * LTS + 2 * lane);
        const uint32_t uv = *reinterpret_cast<const uint32_t*>(oV + r * LTS + 2 * lane);
        k0 += bf16_lo(uk); k1 += bf16_hi(uk); v0 += bf16_lo(uv); v1 += bf16_hi(uv);
      }
      atomicAdd(dbias + E + h * LDH + 2 * lane, k0);
      atomicAdd(dbias + E + h * LDH + 2 * lane + 1, k1);
      atomicAdd(dbias + 2 * E + h * LDH + 2 * lane, v0);
      atomicAdd(dbias + 2 * E + h * LDH + 2 * lane + 1, v1);
    }
  }
}

// host launcher used by tnr_attn_relpos_bwd (attention.cu) for L > 32.  ws: 2 * n_news * A * L floats.
int attn_long_bwd_launch(const void* qkv_bf16, const int64_t* mask, int mask_ld, const float* relbias, const void* dctx_bf16,
                         void* dqkv_bf16, float* dbias, float* ws, int n_news, int L, int A, int E, const tnr_dropout* drop,
                         cudaStream_t st) {
  TNR_REQUIRE(L <= LONG_LMAX, "tnr_attn_relpos_bwd: L=%d exceeds %d (the position table of the encoder)", L, LONG_LMAX);
  TNR_REQUIRE(ws != nullptr, "tnr_attn_relpos_bwd: L=%d > 32 needs a workspace of 2 * n_news * A * L floats", L);
  const int q_blocks = (L + LQB - 1) / LQB;
  const int k_chunks = (L + LKB - 1) / LKB;
  const long long blocks = (long long)n_news * A * q_blocks;
  TNR_REQUIRE(blocks < (1ll << 31), "tnr_attn_relpos_bwd: too many blocks");
  float* ws_lse = ws;
  float* ws_delta = ws + (size_t)n_news * A * L;
  const int smem_dq = 6 * LQB * LTS * 2 + (k_chunks * LKB + 2 * L - 1 + LKB) * 4;
  const int smem_dkv = 8 * LQB * LTS * 2 + (LKB + 2 * L - 1 + LKB) * 4;
  TNR_SET_SMEM(attn_long_bwd_dq_kernel, 6 * LQB * LTS * 2 + (LONG_LMAX + 2 * LONG_LMAX + LKB) * 4);
  TNR_SET_SMEM(attn_long_bwd_dkv_kernel, 8 * LQB * LTS * 2 + (LKB + 2 * LONG_LMAX + LKB) * 4);
  attn_long_bwd_dq_kernel<<<(unsigned)blocks, 128, smem_dq, st>>>(
      reinterpret_cast<const __nv_bfloat16*>(qkv_bf16), mask, mask_ld, relbias, reinterpret_cast<const __nv_bfloat16*>(dctx_bf16),
      reinterpret_cast<__nv_bfloat16*>(dqkv_bf16), dbias, ws_lse, ws_delta, n_news, L, A, E, q_blocks, drop_or_none(drop));
  TNR_LAUNCH_CHECK();
  attn_long_bwd_dkv_kernel<<<(unsigned)blocks, 128, smem_dkv, st>>>(
      reinterpret_cast<const __nv_bfloat16*>(qkv_bf16), mask, mask_ld, relbias, reinterpret_cast<const __nv_bfloat16*>(dctx_bf16),
      reinterpret_cast<__nv_bfloat16*>(dqkv_bf16), dbias, ws_lse, ws_delta, n_news, L, A, E, k_chunks, drop_or_none(drop));
  TNR_LAUNCH_CHECK();
  return 0;
}

int attn_long_q_blocks(int L) { return (L + LQB - 1) / LQB; }

// host launcher used by tnr_attn_relpos_bwd_drel (attention.cu) for L > 32: the same two kernels, the dQ one with the
// diagonal sums.  part: n_news * A * q_blocks * nb floats.
int attn_long_bwd_drel_launch(const void* qkv_bf16, const int64_t* mask, int mask_ld, const float* relbias,
                              const void* dctx_bf16, void* dqkv_bf16, float* dbias, float* ws, int n_news, int L, int A, int E,
                              const tnr_dropout* drop, const int* bucket, int nb, float* part, cudaStream_t st) {
  TNR_REQUIRE(L <= LONG_LMAX, "tnr_attn_relpos_bwd_drel: L=%d exceeds %d", L, LONG_LMAX);
  TNR_REQUIRE(ws != nullptr, "tnr_attn_relpos_bwd_drel: L=%d > 32 needs a workspace of 2 * n_news * A * L floats", L);
  const int q_blocks = (L + LQB - 1) / LQB;
  const int k_chunks = (L + LKB - 1) / LKB;
  const long long blocks = (long long)n_news * A * q_blocks;
  TNR_REQUIRE(blocks < (1ll << 31), "tnr_attn_relpos_bwd_drel: too many blocks");
  float* ws_lse = ws;
  float* ws_delta = ws + (size_t)n_news * A * L;
  const int drel_floats = 8 * L + 4 * 16 * DT_LD;
  const int smem_dq = 6 * LQB * LTS * 2 + (k_chunks * LKB + 2 * L - 1 + LKB + drel_floats) * 4;
  const int smem_dkv = 8 * LQB * LTS * 2 + (LKB + 2 * L - 1 + LKB) * 4;
  TNR_SET_SMEM(attn_long_bwd_dq_drel_kernel,
               6 * LQB * LTS * 2 + (LONG_LMAX + 2 * LONG_LMAX + LKB + 8 * LONG_LMAX + 4 * 16 * DT_LD) * 4);
  TNR_SET_SMEM(attn_long_bwd_dkv_kernel, 8 * LQB * LTS * 2 + (LKB + 2 * LONG_LMAX + LKB) * 4);
  attn_long_bwd_dq_drel_kernel<<<(unsigned)blocks, 128, smem_dq, st>>>(
      reinterpret_cast<const __nv_bfloat16*>(qkv_bf16), mask, mask_ld, relbias, reinterpret_cast<const __nv_bfloat16*>(dctx_bf16),
      reinterpret_cast<__nv_bfloat16*>(dqkv_bf16), dbias, ws_lse, ws_delta, n_news, L, A, E, q_blocks, drop_or_none(drop), bucket,
      nb, part);
  TNR_LAUNCH_CHECK();
  attn_long_bwd_dkv_kernel<<<(unsigned)blocks, 128, smem_dkv, st>>>(
      reinterpret_cast<const __nv_bfloat16*>(qkv_bf16), mask, mask_ld, relbias, reinterpret_cast<const __nv_bfloat16*>(dctx_bf16),
      reinterpret_cast<__nv_bfloat16*>(dqkv_bf16), dbias, ws_lse, ws_delta, n_news, L, A, E, k_chunks, drop_or_none(drop));
  TNR_LAUNCH_CHECK();
  return 0;
}

// host launcher used by tnr_attn_relpos_fwd (attention.cu) for L > 32
int attn_long_fwd_launch(const void* qkv_bf16, const int64_t* mask, int mask_ld, const float* relbias, void* ctx_bf16,
                         int n_news, int L, int A, int E, const tnr_dropout* drop, cudaStream_t st) {
  TNR_REQUIRE(L <= LONG_LMAX, "tnr_attn_relpos_fwd: L=%d exceeds %d (the position table of the encoder)", L, LONG_LMAX);
  const int q_blocks = (L + LQB - 1) / LQB;
  const int k_chunks = (L + LKB - 1) / LKB;
  const long long blocks = (long long)n_news * A * q_blocks;
  TNR_REQUIRE(blocks < (1ll << 31), "tnr_attn_relpos_fwd: too many blocks");
  const int smem = 5 * LQB * LTS * 2 + (k_chunks * LKB + 2 * L - 1 + LKB) * 4;
  TNR_SET_SMEM(attn_long_fwd_kernel, 5 * LQB * LTS * 2 + (LONG_LMAX + 2 * LONG_LMAX + LKB) * 4);
  attn_long_fwd_kernel<<<(unsigned)blocks, 128, smem, st>>>(
      reinterpret_cast<const __nv_bfloat16*>(qkv_bf16), mask, mask_ld, relbias, reinterpret_cast<__nv_bfloat16*>(ctx_bf16),
      n_news, L, A, E, q_blocks, drop_or_none(drop));
  TNR_LAUNCH_CHECK();
  return 0;
}

}  // namespace tnr
