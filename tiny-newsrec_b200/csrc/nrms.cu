// NRMS user encoder: the multi-head self-attention that sits in front of the additive pooling when
// args.model == 'NRMS' (Tiny-NewsRec/model_bert.py:37-100, wired in at :145-148, :162-164, :171-173).
//
//   x'      = v * m + pad_doc * (1 - m)                 (only when user_log_mask is False, :169-170)
//   Q,K,V   = x' W^T + b                                (tnr_sgemm_nt, three planes [3][B*H][Dh])
//   s_ij    = exp(q_i . k_j / sqrt(16)) [* m_j]         (NOT a softmax: no max subtraction, :53-57)
//   ctx_i   = sum_j s_ij v_j / (sum_j s_ij + 1e-8)      (:59-60), heads concatenated (:98)
//
// All fp32 (the head of the model is fp32 end to end).  d_k = d_v = 16 are hard-wired in the reference
// (:146).  H <= 64: one block per impression, one warp per head.  64 < H <= 512: one block per (impression,
// head), whose eight warps share that head's K and V (and q / 4, dctx in the backward) -- 64 KB (forward) and
// 134 KB (backward) of shared memory at H = 512.  Either way a lane owns a query row (forward and the dQ pass of the
// backward) or a key row (the dK / dV pass), so every shared-memory read in the inner loops is a broadcast and nothing
// is reduced across lanes.  The backward recomputes the scores.
// tnr_sgemm_nn is the one GEMM shape the head did not have yet: dX' = dQ W_Q + dK W_K + dV W_V.
#include "common.cuh"

namespace tnr {

constexpr int NR_HMAX = 64;        // longest history of the warp-per-head kernels (user_log_length is 50 in the demo)
constexpr int NR_HLONG = 512;      // history length limit
constexpr int NR_DK = 16;
constexpr int NR_WARPS = 8;
constexpr int NR_THREADS = NR_WARPS * 32;

__device__ __forceinline__ void ld16(float (&r)[NR_DK], const float* p) {
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    const float4 t = *reinterpret_cast<const float4*>(p + 4 * c);
    r[4 * c] = t.x; r[4 * c + 1] = t.y; r[4 * c + 2] = t.z; r[4 * c + 3] = t.w;
  }
}
__device__ __forceinline__ void st16(float* p, const float (&r)[NR_DK]) {
#pragma unroll
  for (int c = 0; c < 4; ++c) *reinterpret_cast<float4*>(p + 4 * c) = make_float4(r[4 * c], r[4 * c + 1], r[4 * c + 2], r[4 * c + 3]);
}
__device__ __forceinline__ float dot16(const float (&a)[NR_DK], const float* b) {
  float s = 0.f;
#pragma unroll
  for (int c = 0; c < NR_DK; ++c) s = fmaf(a[c], b[c], s);
  return s;
}

// ctx_i of one head for the query row at qrow; keys and values [H][16] and the key mask in shared memory
__device__ __forceinline__ void nrms_ctx_row(const float* qrow, const float* sk, const float* sv, const float* smk, int H,
                                             float* out) {
  float qi[NR_DK], acc[NR_DK];
  ld16(qi, qrow);
#pragma unroll
  for (int c = 0; c < NR_DK; ++c) { qi[c] *= 0.25f; acc[c] = 0.f; }      // 1 / sqrt(d_k), exact
  float sum = 0.f;
  for (int j = 0; j < H; ++j) {
    const float s = expf(dot16(qi, sk + j * NR_DK)) * smk[j];
    sum += s;
#pragma unroll
    for (int c = 0; c < NR_DK; ++c) acc[c] = fmaf(s, sv[j * NR_DK + c], acc[c]);
  }
  const float inv = 1.0f / (sum + 1e-8f);
#pragma unroll
  for (int c = 0; c < NR_DK; ++c) acc[c] *= inv;
  st16(out, acc);
}

// backward pass 1, query row i: dq_i, 1 / Z_i and D_i (sq holds q / 4, sd dctx)
__device__ __forceinline__ void nrms_dq_row(int i, const float* sq, const float* sk, const float* sv, const float* sd,
                                            const float* smk, int H, float* dq_out, float* sZ, float* sD) {
  float qi[NR_DK], di[NR_DK], acc[NR_DK];
  ld16(qi, sq + i * NR_DK);
  ld16(di, sd + i * NR_DK);
#pragma unroll
  for (int c = 0; c < NR_DK; ++c) acc[c] = 0.f;
  float sum = 0.f;
  for (int j = 0; j < H; ++j) {
    const float s = expf(dot16(qi, sk + j * NR_DK)) * smk[j];
    sum += s;
#pragma unroll
    for (int c = 0; c < NR_DK; ++c) acc[c] = fmaf(s, sv[j * NR_DK + c], acc[c]);
  }
  const float inv = 1.0f / (sum + 1e-8f);
  float Di = 0.f;
#pragma unroll
  for (int c = 0; c < NR_DK; ++c) Di = fmaf(di[c], acc[c] * inv, Di);
#pragma unroll
  for (int c = 0; c < NR_DK; ++c) acc[c] = 0.f;
  for (int j = 0; j < H; ++j) {
    const float a = expf(dot16(qi, sk + j * NR_DK)) * smk[j] * inv;
    const float dl = a * (dot16(di, sv + j * NR_DK) - Di);
#pragma unroll
    for (int c = 0; c < NR_DK; ++c) acc[c] = fmaf(dl, sk[j * NR_DK + c], acc[c]);
  }
#pragma unroll
  for (int c = 0; c < NR_DK; ++c) acc[c] *= 0.25f;
  st16(dq_out, acc);
  sZ[i] = inv;
  sD[i] = Di;
}

// backward pass 2, key row j: dk_j, dv_j (needs sZ / sD of every query row)
__device__ __forceinline__ void nrms_dkv_row(int j, const float* sq, const float* sk, const float* sv, const float* sd,
                                             const float* sZ, const float* sD, const float* smk, int H, float* dk_out,
                                             float* dv_out) {
  float kj[NR_DK], vj[NR_DK], gk[NR_DK], gv[NR_DK];
  ld16(kj, sk + j * NR_DK);
  ld16(vj, sv + j * NR_DK);
#pragma unroll
  for (int c = 0; c < NR_DK; ++c) { gk[c] = 0.f; gv[c] = 0.f; }
  const float mj = smk[j];
  for (int i = 0; i < H; ++i) {
    const float a = expf(dot16(kj, sq + i * NR_DK)) * mj * sZ[i];
    const float dl = a * (dot16(vj, sd + i * NR_DK) - sD[i]);
#pragma unroll
    for (int c = 0; c < NR_DK; ++c) {
      gv[c] = fmaf(a, sd[i * NR_DK + c], gv[c]);
      gk[c] = fmaf(dl, sq[i * NR_DK + c], gk[c]);     // sq already carries the 1/4
    }
  }
  st16(dk_out, gk);
  st16(dv_out, gv);
}

// stage rows [H][16] of head column col: k / v (and q / 4, dctx when sq != nullptr), threads tid0, tid0 + step, ...
__device__ __forceinline__ void nrms_stage(const float* q, const float* k, const float* v, const float* dctx, float* sq,
                                           float* sk, float* sv, float* sd, size_t row0, int H, int Dh, int col, int tid0,
                                           int step) {
  for (int i = tid0; i < H * 4; i += step) {
    const int r = i >> 2, c = (i & 3) * 4;
    const size_t g = (row0 + r) * Dh + col + c;
    *reinterpret_cast<float4*>(sk + r * NR_DK + c) = *reinterpret_cast<const float4*>(k + g);
    *reinterpret_cast<float4*>(sv + r * NR_DK + c) = *reinterpret_cast<const float4*>(v + g);
    if (sq != nullptr) {
      float4 t = *reinterpret_cast<const float4*>(q + g);
      t.x *= 0.25f; t.y *= 0.25f; t.z *= 0.25f; t.w *= 0.25f;
      *reinterpret_cast<float4*>(sq + r * NR_DK + c) = t;
      *reinterpret_cast<float4*>(sd + r * NR_DK + c) = *reinterpret_cast<const float4*>(dctx + g);
    }
  }
}

// ---------------------------------------------------------------- pad_doc blend (user_log_mask = False)
__global__ void __launch_bounds__(256)
nrms_blend_fwd_kernel(const float* __restrict__ vecs, const float* __restrict__ mask, const float* __restrict__ pad,
                      float* __restrict__ out, long long n4, int D4) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n4) return;
  const long long r = i / D4;
  const int c = (int)(i - r * D4);
  const float m = mask[r];
  const float4 v = reinterpret_cast<const float4*>(vecs)[i];
  const float4 p = reinterpret_cast<const float4*>(pad)[c];
  const float om = 1.0f - m;
  reinterpret_cast<float4*>(out)[i] = make_float4(v.x * m + p.x * om, v.y * m + p.y * om, v.z * m + p.z * om, v.w * m + p.w * om);
}

// d_vecs[r] += d_blend[r] * m_r ; dpad += sum_r d_blend[r] (1 - m_r).  mask == nullptr: plain accumulate.
constexpr int NB_ROWS = 16;
__global__ void __launch_bounds__(256)
nrms_blend_bwd_kernel(const float* __restrict__ db, const float* __restrict__ mask, float* __restrict__ d_vecs,
                      float* __restrict__ dpad, int rows, int D) {
  const int r0 = blockIdx.x * NB_ROWS;
  for (int d = threadIdx.x; d < D; d += blockDim.x) {
    float gp = 0.f;
    for (int r = r0; r < min(r0 + NB_ROWS, rows); ++r) {
      const float g = db[(size_t)r * D + d];
      if (mask) {
        const float m = mask[r];
        d_vecs[(size_t)r * D + d] += g * m;
        gp = fmaf(g, 1.0f - m, gp);
      } else {
        d_vecs[(size_t)r * D + d] += g;
      }
    }
    if (mask && dpad) atomicAdd(dpad + d, gp);
  }
}

// ---------------------------------------------------------------- attention forward
__global__ void __launch_bounds__(NR_THREADS)
nrms_attn_fwd_kernel(const float* __restrict__ q, const float* __restrict__ k, const float* __restrict__ v,
                     const float* __restrict__ mask, float* __restrict__ ctx, int H, int n_heads) {
  extern __shared__ __align__(16) float nr_sm[];
  const int warp = uniform_warp_id(), lane = threadIdx.x & 31, b = blockIdx.x;
  const int Dh = n_heads * NR_DK;
  float* sk = nr_sm + warp * (2 * NR_HMAX * NR_DK);
  float* sv = sk + NR_HMAX * NR_DK;
  float* smk = nr_sm + NR_WARPS * (2 * NR_HMAX * NR_DK);
  for (int j = threadIdx.x; j < H; j += NR_THREADS) smk[j] = mask ? mask[(size_t)b * H + j] : 1.0f;
  __syncthreads();
  const size_t row0 = (size_t)b * H;
  for (int head = warp; head < n_heads; head += NR_WARPS) {
    const int col = head * NR_DK;
    nrms_stage(q, k, v, nullptr, nullptr, sk, sv, nullptr, row0, H, Dh, col, lane, 32);
    __syncwarp();
    for (int i = lane; i < H; i += 32) nrms_ctx_row(q + (row0 + i) * Dh + col, sk, sv, smk, H, ctx + (row0 + i) * Dh + col);
    __syncwarp();
  }
}

// H > 64: block (b, head); the eight warps share the head's K / V
__global__ void __launch_bounds__(NR_THREADS)
nrms_attn_fwd_long_kernel(const float* __restrict__ q, const float* __restrict__ k, const float* __restrict__ v,
                          const float* __restrict__ mask, float* __restrict__ ctx, int H, int n_heads) {
  extern __shared__ __align__(16) float nr_sm[];
  const int b = blockIdx.x, col = blockIdx.y * NR_DK, Dh = n_heads * NR_DK;
  float* sk = nr_sm;                       // [H][16]
  float* sv = sk + H * NR_DK;              // [H][16]
  float* smk = sv + H * NR_DK;             // [H]
  const size_t row0 = (size_t)b * H;
  for (int j = threadIdx.x; j < H; j += NR_THREADS) smk[j] = mask ? mask[row0 + j] : 1.0f;
  nrms_stage(q, k, v, nullptr, nullptr, sk, sv, nullptr, row0, H, Dh, col, threadIdx.x, NR_THREADS);
  __syncthreads();
  for (int i = threadIdx.x; i < H; i += NR_THREADS)
    nrms_ctx_row(q + (row0 + i) * Dh + col, sk, sv, smk, H, ctx + (row0 + i) * Dh + col);
}

// ---------------------------------------------------------------- attention backward (recomputes s)
//   a_ij = s_ij / Z_i,  da_ij = dctx_i . v_j,  D_i = dctx_i . ctx_i,  dl_ij = a_ij (da_ij - D_i)
//   dq_i = sum_j dl_ij k_j / 4,  dk_j = sum_i dl_ij q_i / 4,  dv_j = sum_i a_ij dctx_i
__global__ void __launch_bounds__(NR_THREADS)
nrms_attn_bwd_kernel(const float* __restrict__ q, const float* __restrict__ k, const float* __restrict__ v,
                     const float* __restrict__ mask, const float* __restrict__ dctx, float* __restrict__ dq,
                     float* __restrict__ dk, float* __restrict__ dv, int H, int n_heads) {
  extern __shared__ __align__(16) float nr_sm[];
  const int warp = uniform_warp_id(), lane = threadIdx.x & 31, b = blockIdx.x;
  const int Dh = n_heads * NR_DK;
  constexpr int PER_WARP = 4 * NR_HMAX * NR_DK + 2 * NR_HMAX;
  float* sq = nr_sm + warp * PER_WARP;          // q / 4
  float* sk = sq + NR_HMAX * NR_DK;
  float* sv = sk + NR_HMAX * NR_DK;
  float* sd = sv + NR_HMAX * NR_DK;             // dctx
  float* sZ = sd + NR_HMAX * NR_DK;             // 1 / Z_i
  float* sD = sZ + NR_HMAX;                     // D_i
  float* smk = nr_sm + NR_WARPS * PER_WARP;
  for (int j = threadIdx.x; j < H; j += NR_THREADS) smk[j] = mask ? mask[(size_t)b * H + j] : 1.0f;
  __syncthreads();
  const size_t row0 = (size_t)b * H;
  for (int head = warp; head < n_heads; head += NR_WARPS) {
    const int col = head * NR_DK;
    nrms_stage(q, k, v, dctx, sq, sk, sv, sd, row0, H, Dh, col, lane, 32);
    __syncwarp();
    // pass 1: lane = query row
    for (int i = lane; i < H; i += 32) nrms_dq_row(i, sq, sk, sv, sd, smk, H, dq + (row0 + i) * Dh + col, sZ, sD);
    __syncwarp();
    // pass 2: lane = key row
    for (int j = lane; j < H; j += 32)
      nrms_dkv_row(j, sq, sk, sv, sd, sZ, sD, smk, H, dk + (row0 + j) * Dh + col, dv + (row0 + j) * Dh + col);
    __syncwarp();
  }
}

// H > 64: block (b, head); pass 2 needs 1 / Z_i and D_i of every query row, hence the __syncthreads between the passes
__global__ void __launch_bounds__(NR_THREADS)
nrms_attn_bwd_long_kernel(const float* __restrict__ q, const float* __restrict__ k, const float* __restrict__ v,
                          const float* __restrict__ mask, const float* __restrict__ dctx, float* __restrict__ dq,
                          float* __restrict__ dk, float* __restrict__ dv, int H, int n_heads) {
  extern __shared__ __align__(16) float nr_sm[];
  const int b = blockIdx.x, col = blockIdx.y * NR_DK, Dh = n_heads * NR_DK;
  float* sq = nr_sm;                       // [H][16] q / 4
  float* sk = sq + H * NR_DK;
  float* sv = sk + H * NR_DK;
  float* sd = sv + H * NR_DK;              // dctx
  float* sZ = sd + H * NR_DK;              // [H] 1 / Z_i
  float* sD = sZ + H;                      // [H] D_i
  float* smk = sD + H;                     // [H]
  const size_t row0 = (size_t)b * H;
  for (int j = threadIdx.x; j < H; j += NR_THREADS) smk[j] = mask ? mask[row0 + j] : 1.0f;
  nrms_stage(q, k, v, dctx, sq, sk, sv, sd, row0, H, Dh, col, threadIdx.x, NR_THREADS);
  __syncthreads();
  for (int i = threadIdx.x; i < H; i += NR_THREADS) nrms_dq_row(i, sq, sk, sv, sd, smk, H, dq + (row0 + i) * Dh + col, sZ, sD);
  __syncthreads();
  for (int j = threadIdx.x; j < H; j += NR_THREADS)
    nrms_dkv_row(j, sq, sk, sv, sd, sZ, sD, smk, H, dk + (row0 + j) * Dh + col, dv + (row0 + j) * Dh + col);
}

// ---------------------------------------------------------------- C[M,N] = sum_p A_p[M,K] . B_p[K,N]
// 64 x 64 tiles, 4 warps, TF32 mma.sync with cvt.rna inputs and fp32 accumulate (as tnr_sgemm_nt / tn).
constexpr int SN_T = 64, SN_K = 32, SN_THREADS = 128;
__device__ __forceinline__ uint32_t nn_tf32(float x) { return __float_as_uint(x) + 0x1000u; }   // = cvt.rna (head_mma.cu)
__device__ __forceinline__ void nn_cp16(void* smem_dst, const void* src, bool valid) {
  const uint32_t dst = (uint32_t)__cvta_generic_to_shared(smem_dst);
  const int bytes = valid ? 16 : 0;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(bytes) : "memory");
}

__global__ void __launch_bounds__(SN_THREADS)
sgemm_nn_kernel(const float* __restrict__ A, const float* __restrict__ Bm, float* __restrict__ C, int M, int N, int K,
                int parts, long long sA, long long sB) {
  __shared__ __align__(16) float As[2][SN_T][SN_K + 4];
  __shared__ __align__(16) float Bs[2][SN_K][SN_T + 8];
  const int tid = threadIdx.x, warp = uniform_warp_id(), lane = tid & 31, g = lane >> 2, t = lane & 3;
  const int wm = warp >> 1, wn = warp & 1;
  const int m0 = blockIdx.y * SN_T, n0 = blockIdx.x * SN_T;
  float acc[2][4][4] = {};
  const int nk = (K + SN_K - 1) / SN_K;
  const int total = nk * parts;
  auto load = [&](int st, int kc) {
    const int p = kc / nk, k0 = (kc - p * nk) * SN_K;
    const float* Ap = A + p * sA;
    const float* Bp = Bm + p * sB;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int idx = tid + i * SN_THREADS;
      {
        const int r = idx >> 3, c4 = (idx & 7) * 4;
        const bool va = (k0 + c4 + 4 <= K) && (m0 + r < M);
        nn_cp16(&As[st][r][c4], va ? Ap + (size_t)(m0 + r) * K + k0 + c4 : Ap, va);
      }
      {
        const int r = idx >> 4, c4 = (idx & 15) * 4;
        const bool vb = (k0 + r < K) && (n0 + c4 + 4 <= N);
        nn_cp16(&Bs[st][r][c4], vb ? Bp + (size_t)(k0 + r) * N + n0 + c4 : Bp, vb);
      }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  load(0, 0);
  for (int kc = 0; kc < total; ++kc) {
    const int st = kc & 1;
    if (kc + 1 < total) { load(st ^ 1, kc + 1); asm volatile("cp.async.wait_group 1;" ::: "memory"); }
    else { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
    __syncthreads();
#pragma unroll
    for (int ks = 0; ks < SN_K / 8; ++ks) {
      uint32_t bf[4][2];
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) {
        bf[nt][0] = nn_tf32(Bs[st][ks * 8 + t][wn * 32 + nt * 8 + g]);
        bf[nt][1] = nn_tf32(Bs[st][ks * 8 + t + 4][wn * 32 + nt * 8 + g]);
      }
#pragma unroll
      for (int mt = 0; mt < 2; ++mt) {
        uint32_t a[4];
        const int r = wm * 32 + mt * 16 + g;
        a[0] = nn_tf32(As[st][r][ks * 8 + t]);
        a[1] = nn_tf32(As[st][r + 8][ks * 8 + t]);
        a[2] = nn_tf32(As[st][r][ks * 8 + t + 4]);
        a[3] = nn_tf32(As[st][r + 8][ks * 8 + t + 4]);
#pragma unroll
        for (int nt = 0; nt < 4; ++nt)
          asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                       : "+f"(acc[mt][nt][0]), "+f"(acc[mt][nt][1]), "+f"(acc[mt][nt][2]), "+f"(acc[mt][nt][3])
                       : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(bf[nt][0]), "r"(bf[nt][1]));
      }
    }
    __syncthreads();
  }
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < 4; ++nt)
#pragma unroll
      for (int hi = 0; hi < 2; ++hi) {
        const int m = m0 + wm * 32 + mt * 16 + g + hi * 8;
        if (m >= M) continue;
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int n = n0 + wn * 32 + nt * 8 + 2 * t + e;
          if (n < N) C[(size_t)m * N + n] = acc[mt][nt][hi * 2 + e];
        }
      }
}

}  // namespace tnr

using namespace tnr;

#define TNR_API extern "C" __attribute__((visibility("default")))

static int nrms_check(const char* who, int H, int n_heads) {
  TNR_REQUIRE(H >= 1 && H <= NR_HLONG, "%s: history length %d not supported (1..%d)", who, H, NR_HLONG);
  TNR_REQUIRE(n_heads >= 1 && n_heads <= 64, "%s: n_heads=%d out of range (1..64)", who, n_heads);
  return 0;
}

TNR_API int tnr_nrms_blend_fwd(const float* vecs, const float* mask, const float* pad_doc, float* out, int rows, int D,
                               void* stream) {
  TNR_REQUIRE(D % 4 == 0 && D > 0, "tnr_nrms_blend_fwd: D=%d must be a positive multiple of 4", D);
  TNR_REQUIRE(((uintptr_t)vecs | (uintptr_t)pad_doc | (uintptr_t)out) % 16 == 0, "tnr_nrms_blend_fwd: 16-byte alignment required");
  if (rows == 0) return 0;
  const long long n4 = (long long)rows * (D / 4);
  nrms_blend_fwd_kernel<<<(unsigned)((n4 + 255) / 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(vecs, mask, pad_doc, out, n4, D / 4);
  TNR_LAUNCH_CHECK();
  return 0;
}

TNR_API int tnr_nrms_blend_bwd(const float* d_blend, const float* mask, float* d_vecs, float* dpad, int rows, int D,
                               void* stream) {
  TNR_REQUIRE(D > 0, "tnr_nrms_blend_bwd: D=%d", D);
  if (rows == 0) return 0;
  nrms_blend_bwd_kernel<<<(rows + NB_ROWS - 1) / NB_ROWS, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(d_blend, mask, d_vecs, dpad, rows, D);
  TNR_LAUNCH_CHECK();
  return 0;
}

TNR_API int tnr_nrms_attn_fwd(const float* q, const float* k, const float* v, const float* mask, float* ctx, int B, int H,
                              int n_heads, void* stream) {
  if (nrms_check("tnr_nrms_attn_fwd", H, n_heads)) return 1;
  TNR_REQUIRE(((uintptr_t)q | (uintptr_t)k | (uintptr_t)v | (uintptr_t)ctx) % 16 == 0, "tnr_nrms_attn_fwd: 16-byte alignment required");
  if (B == 0) return 0;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (H <= NR_HMAX) {
    const int smem = (NR_WARPS * 2 * NR_HMAX * NR_DK + NR_HMAX) * 4;
    TNR_SET_SMEM(nrms_attn_fwd_kernel, smem);
    nrms_attn_fwd_kernel<<<B, NR_THREADS, smem, st>>>(q, k, v, mask, ctx, H, n_heads);
  } else {
    const int smem = (2 * H * NR_DK + H) * 4;
    TNR_SET_SMEM(nrms_attn_fwd_long_kernel, smem);
    nrms_attn_fwd_long_kernel<<<dim3(B, n_heads), NR_THREADS, smem, st>>>(q, k, v, mask, ctx, H, n_heads);
  }
  TNR_LAUNCH_CHECK();
  return 0;
}

TNR_API int tnr_nrms_attn_bwd(const float* q, const float* k, const float* v, const float* mask, const float* d_ctx,
                              float* dq, float* dk, float* dv, int B, int H, int n_heads, void* stream) {
  if (nrms_check("tnr_nrms_attn_bwd", H, n_heads)) return 1;
  TNR_REQUIRE(((uintptr_t)q | (uintptr_t)k | (uintptr_t)v | (uintptr_t)d_ctx | (uintptr_t)dq | (uintptr_t)dk | (uintptr_t)dv) % 16 == 0,
              "tnr_nrms_attn_bwd: 16-byte alignment required");
  if (B == 0) return 0;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (H <= NR_HMAX) {
    const int smem = (NR_WARPS * (4 * NR_HMAX * NR_DK + 2 * NR_HMAX) + NR_HMAX) * 4;
    TNR_SET_SMEM(nrms_attn_bwd_kernel, smem);
    nrms_attn_bwd_kernel<<<B, NR_THREADS, smem, st>>>(q, k, v, mask, d_ctx, dq, dk, dv, H, n_heads);
  } else {
    const int smem = (4 * H * NR_DK + 3 * H) * 4;
    TNR_SET_SMEM(nrms_attn_bwd_long_kernel, smem);
    nrms_attn_bwd_long_kernel<<<dim3(B, n_heads), NR_THREADS, smem, st>>>(q, k, v, mask, d_ctx, dq, dk, dv, H, n_heads);
  }
  TNR_LAUNCH_CHECK();
  return 0;
}

TNR_API int tnr_sgemm_nn(const float* A, const float* Bm, float* C, int M, int N, int K, int parts, long long sA,
                         long long sB, void* stream) {
  TNR_REQUIRE(K % 4 == 0 && N % 4 == 0, "tnr_sgemm_nn: K=%d and N=%d must be multiples of 4", K, N);
  TNR_REQUIRE(((uintptr_t)A % 16 == 0) && ((uintptr_t)Bm % 16 == 0) && sA % 4 == 0 && sB % 4 == 0,
              "tnr_sgemm_nn: operands must be 16-byte aligned");
  TNR_REQUIRE(parts >= 1 && K >= 4, "tnr_sgemm_nn: parts=%d, K=%d", parts, K);
  if (M == 0 || N == 0) return 0;
  dim3 grid((N + SN_T - 1) / SN_T, (M + SN_T - 1) / SN_T, 1);
  sgemm_nn_kernel<<<grid, SN_THREADS, 0, reinterpret_cast<cudaStream_t>(stream)>>>(A, Bm, C, M, N, K, parts, sA, sB);
  TNR_LAUNCH_CHECK();
  return 0;
}
