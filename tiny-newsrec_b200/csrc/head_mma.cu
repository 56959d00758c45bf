// fp32 "head" GEMM-shaped work on the warp-level tensor path (mma.sync m16n8k8, TF32 inputs
// rounded with cvt.rna, fp32 accumulate): the additive-attention user encoders (student + M
// teachers in ONE launch), the student user-encoder backward, and the two small batched fp32
// GEMMs of the per-teacher projection (transform_matrix forward / weight gradient).
// These are a few MFLOP..GFLOP per step on [B*H, 256] fp32 matrices: far below a tcgen05 tile
// economy, but they must not serialise on 32 blocks either -- every kernel here spreads over
// >= 148 CTAs or finishes in a few microseconds.
//
// Reference: Tiny-NewsRec/model_bert.py:155-176 (UserEncoder, NAML branches), :15-34
// (AttentionPooling), :277-278,283 (transform_matrix), and their autograd backward.
#include "common.cuh"
#include "tc_ptx.cuh"

namespace tnr {

// fp32 -> TF32, round to nearest (ties away), as cvt.rna.tf32.f32 -- which ptxas expands to ~8 instructions on
// sm_100 (FSETP |x| < inf, three PLOP3, a predicated IADD, LOP3).  Adding half a TF32 ulp to the magnitude bits is
// the same rounding for every finite input (inf stays inf, NaN stays NaN) and the tensor core ignores the low 13
// bits of a .tf32 operand, so one IADD does it.
__device__ __forceinline__ uint32_t f2tf32(float x) { return __float_as_uint(x) + 0x1000u; }
// tanh(x) = 1 - 2 / (1 + e^{2x}): 5 instructions against ~25 for tanhf (64 evaluations per thread made the
// epilogue a third of the kernel); absolute error < 3e-7, saturates to +-1 exactly for large |x|.
__device__ __forceinline__ float tanh_exp(float x) {
  return 1.0f - __fdividef(2.0f, 1.0f + __expf(2.0f * x));
}
__device__ __forceinline__ void mma_tf32(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
// 3xTF32 split of an fp32 operand for the fp32 inference mode: hi = tf32_rn(x) as a MASKED float, so lo = x - hi is
// exact; lo goes to the tensor core as f2tf32(lo).  hi + tf32(lo) carries ~21 of x's 24 significand bits.
__device__ __forceinline__ void split_tf32(float x, uint32_t& hi, uint32_t& lo) {
  hi = (__float_as_uint(x) + 0x1000u) & 0xffffe000u;
  lo = f2tf32(x - __uint_as_float(hi));
}
// c += a b to ~fp32 accuracy from split operands: lo_a hi_b and hi_a lo_b first (the small terms), then hi_a hi_b.
// The dropped lo_a lo_b term is ~2^-22 of the product.
__device__ __forceinline__ void mma_tf32x3(float (&c)[4], const uint32_t (&ah)[4], const uint32_t (&al)[4], uint32_t bh0,
                                           uint32_t bh1, uint32_t bl0, uint32_t bl1) {
  mma_tf32(c, al, bh0, bh1);
  mma_tf32(c, ah, bl0, bl1);
  mma_tf32(c, ah, bh0, bh1);
}
__device__ __forceinline__ void cp_async16_zfill(void* smem_dst, const void* src, bool valid) {
  const uint32_t dst = (uint32_t)__cvta_generic_to_shared(smem_dst);
  const int bytes = valid ? 16 : 0;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// ----------------------------------------------------------------------------------
// batched fp32 GEMMs, 64 x 64 tiles, 4 warps (2 x 2), K chunks of 32 double-buffered with cp.async
//   NT: C[b][M,N]   = A[b][M,K] . B[b][N,K]^T + bias[b][N]
//   TN: C[b][N1,N2] += A[b][R,N1]^T . B[b][R,N2];  cbias[b][N1] += colsum(A[b])  (split over R, fp32 atomics)
// ----------------------------------------------------------------------------------
constexpr int SG_T = 64, SG_K = 32, SG_THREADS = 128;

// SPLIT: the fp32 inference mode (3xTF32 from the fp32 tiles, three mma.sync per product, see mma_tf32x3)
template <bool SPLIT>
__global__ void __launch_bounds__(SG_THREADS)
sgemm_nt_kernel(const float* __restrict__ A, const float* __restrict__ Bm, const float* __restrict__ bias,
                float* __restrict__ C, int M, int N, int K, long long sA, long long sB, long long sbias, long long sC) {
  __shared__ __align__(16) float As[2][SG_T][SG_K + 4];
  __shared__ __align__(16) float Bs[2][SG_T][SG_K + 4];
  A += blockIdx.z * sA; Bm += blockIdx.z * sB; C += blockIdx.z * sC;
  if (bias) bias += blockIdx.z * sbias;
  const int tid = threadIdx.x, warp = uniform_warp_id(), lane = tid & 31, g = lane >> 2, t = lane & 3;
  const int wm = warp >> 1, wn = warp & 1;
  const int m0 = blockIdx.y * SG_T, n0 = blockIdx.x * SG_T;
  float acc[2][4][4] = {};
  const int nk = (K + SG_K - 1) / SG_K;
  auto load = [&](int st, int kc) {
    const int k0 = kc * SG_K;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int idx = tid + i * SG_THREADS, r = idx >> 3, c4 = (idx & 7) * 4;
      const bool kv = k0 + c4 + 4 <= K;
      const bool va = kv && (m0 + r < M), vb = kv && (n0 + r < N);
      cp_async16_zfill(&As[st][r][c4], va ? A + (size_t)(m0 + r) * K + k0 + c4 : A, va);
      cp_async16_zfill(&Bs[st][r][c4], vb ? Bm + (size_t)(n0 + r) * K + k0 + c4 : Bm, vb);
    }
    cp_async_commit();
  };
  load(0, 0);
  for (int kc = 0; kc < nk; ++kc) {
    const int st = kc & 1;
    if (kc + 1 < nk) { load(st ^ 1, kc + 1); cp_async_wait<1>(); } else { cp_async_wait<0>(); }
    __syncthreads();
#pragma unroll
    for (int ks = 0; ks < SG_K / 8; ++ks) {
      if constexpr (SPLIT) {
        uint32_t bh[4][2], bl[4][2];
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
          split_tf32(Bs[st][wn * 32 + nt * 8 + g][ks * 8 + t], bh[nt][0], bl[nt][0]);
          split_tf32(Bs[st][wn * 32 + nt * 8 + g][ks * 8 + t + 4], bh[nt][1], bl[nt][1]);
        }
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
          uint32_t ah[4], al[4];
          const int r = wm * 32 + mt * 16 + g;
          split_tf32(As[st][r][ks * 8 + t], ah[0], al[0]);
          split_tf32(As[st][r + 8][ks * 8 + t], ah[1], al[1]);
          split_tf32(As[st][r][ks * 8 + t + 4], ah[2], al[2]);
          split_tf32(As[st][r + 8][ks * 8 + t + 4], ah[3], al[3]);
#pragma unroll
          for (int nt = 0; nt < 4; ++nt) mma_tf32x3(acc[mt][nt], ah, al, bh[nt][0], bh[nt][1], bl[nt][0], bl[nt][1]);
        }
      } else {
        uint32_t b[4][2];
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
          b[nt][0] = f2tf32(Bs[st][wn * 32 + nt * 8 + g][ks * 8 + t]);
          b[nt][1] = f2tf32(Bs[st][wn * 32 + nt * 8 + g][ks * 8 + t + 4]);
        }
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
          uint32_t a[4];
          const int r = wm * 32 + mt * 16 + g;
          a[0] = f2tf32(As[st][r][ks * 8 + t]);
          a[1] = f2tf32(As[st][r + 8][ks * 8 + t]);
          a[2] = f2tf32(As[st][r][ks * 8 + t + 4]);
          a[3] = f2tf32(As[st][r + 8][ks * 8 + t + 4]);
#pragma unroll
          for (int nt = 0; nt < 4; ++nt) mma_tf32(acc[mt][nt], a, b[nt][0], b[nt][1]);
        }
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
          if (n < N) C[(size_t)m * N + n] = acc[mt][nt][hi * 2 + e] + (bias ? bias[n] : 0.f);
        }
      }
}

__global__ void __launch_bounds__(SG_THREADS)
sgemm_tn_kernel(const float* __restrict__ A, const float* __restrict__ Bm, float* __restrict__ C, float* __restrict__ cbias,
                int R, int N1, int N2, int splits, int rows_per_split, long long sA, long long sB, long long sC,
                long long sbias) {
  __shared__ __align__(16) float As[2][SG_K][SG_T + 8];
  __shared__ __align__(16) float Bs[2][SG_K][SG_T + 8];
  const int batch = blockIdx.z / splits, split = blockIdx.z - batch * splits;
  A += batch * sA; Bm += batch * sB; C += batch * sC;
  if (cbias) cbias += batch * sbias;
  const int tid = threadIdx.x, warp = uniform_warp_id(), lane = tid & 31, g = lane >> 2, t = lane & 3;
  const int wm = warp >> 1, wn = warp & 1;
  const int i0 = blockIdx.y * SG_T, j0 = blockIdx.x * SG_T;
  const int r_begin = split * rows_per_split;
  const int r_end = min(R, r_begin + rows_per_split);
  float acc[2][4][4] = {};
  float bsum = 0.f;
  const int nk = (r_end - r_begin + SG_K - 1) / SG_K;
  auto load = [&](int st, int kc) {
    const int r0 = r_begin + kc * SG_K;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int idx = tid + i * SG_THREADS, r = idx >> 4, c4 = (idx & 15) * 4;
      const bool rv = r0 + r < r_end;
      const bool va = rv && (i0 + c4 + 4 <= N1), vb = rv && (j0 + c4 + 4 <= N2);
      cp_async16_zfill(&As[st][r][c4], va ? A + (size_t)(r0 + r) * N1 + i0 + c4 : A, va);
      cp_async16_zfill(&Bs[st][r][c4], vb ? Bm + (size_t)(r0 + r) * N2 + j0 + c4 : Bm, vb);
    }
    cp_async_commit();
  };
  if (nk > 0) load(0, 0);
  for (int kc = 0; kc < nk; ++kc) {
    const int st = kc & 1;
    if (kc + 1 < nk) { load(st ^ 1, kc + 1); cp_async_wait<1>(); } else { cp_async_wait<0>(); }
    __syncthreads();
    if (cbias != nullptr && blockIdx.x == 0 && tid < SG_T) {
#pragma unroll 8
      for (int r = 0; r < SG_K; ++r) bsum += As[st][r][tid];
    }
#pragma unroll
    for (int ks = 0; ks < SG_K / 8; ++ks) {
      uint32_t b[4][2];
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) {
        b[nt][0] = f2tf32(Bs[st][ks * 8 + t][wn * 32 + nt * 8 + g]);
        b[nt][1] = f2tf32(Bs[st][ks * 8 + t + 4][wn * 32 + nt * 8 + g]);
      }
#pragma unroll
      for (int mt = 0; mt < 2; ++mt) {
        uint32_t a[4];
        const int m = wm * 32 + mt * 16 + g;
        a[0] = f2tf32(As[st][ks * 8 + t][m]);
        a[1] = f2tf32(As[st][ks * 8 + t][m + 8]);
        a[2] = f2tf32(As[st][ks * 8 + t + 4][m]);
        a[3] = f2tf32(As[st][ks * 8 + t + 4][m + 8]);
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) mma_tf32(acc[mt][nt], a, b[nt][0], b[nt][1]);
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
        const int m = i0 + wm * 32 + mt * 16 + g + hi * 8;
        if (m >= N1) continue;
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int n = j0 + wn * 32 + nt * 8 + 2 * t + e;
          if (n < N2) atomicAdd(C + (size_t)m * N2 + n, acc[mt][nt][hi * 2 + e]);
        }
      }
  if (cbias != nullptr && blockIdx.x == 0 && tid < SG_T && i0 + tid < N1) atomicAdd(cbias + i0 + tid, bsum);
}

// ----------------------------------------------------------------------------------
// user encoders, forward.  grid (B, n_enc): block (b, i) handles impression b of encoder i.
//   blend (use_mask == 0): v = vec*m + pad_doc*(1-m); alpha unmasked
//   mask  (use_mask == 1): v = vec;  alpha *= m
//   e = tanh(v W1^T + b1) [H, Q] (TF32 mma); alpha = exp(e.w2 + b2)
//   a = alpha / (sum + 1e-8); user = sum_h a_h v_h   (fp32)
// W1 is streamed through shared memory in 16-column chunks (cp.async, double buffered; ~100 KB per block so two
// blocks share an SM and one computes while the other waits).  v1 pulled the W1 fragments straight from L2 into
// registers one k-step ahead: a dependent ~700-cycle load per k-step made the eval-scoring launch (4 096
// impressions) latency-bound at 519 us.  With `idx` the history rows are gathered from the news table inside the
// kernel (run.py:340-343 reads news_scoring[idx] and feeds the user encoder): no [B,H,D] intermediate.
// ----------------------------------------------------------------------------------
constexpr int UE_THREADS = 256;
constexpr int UE_HMAX = 64;           // history rows of one tile; longer histories take the chunked (LONG) kernels
constexpr int UE_HLONG = 512;         // history length limit (user_log_length)
constexpr int UE_MAX_ENC = 9;
constexpr int UE_KC = 16;             // W1 chunk width (k)
constexpr int UE_WS = UE_KC + 4;      // padded chunk row: conflict-free fragment reads

struct UeFwdParams {
  tnr_user_encoder_io enc[UE_MAX_ENC];
  const float* mask;
  const int32_t* idx;                 // optional [B,H] row ids into enc[*].vecs (then a [n_rows, D] table)
  long long n_rows;
  int use_mask, H, D, Q;
};

// Histories longer than 64 rows (LONG = true, 64 < H <= 512) walk the history in 64-row chunks with the same tile
// body: each chunk is staged, multiplied against the re-streamed W1 (re-read from L2 once per chunk) and leaves its
// logits in slog[H]; the softmax and the weighted sum then run once over all H rows.  H <= 64 is one chunk (LONG =
// false compiles to the single-tile kernel).
// SPLIT = true is the fp32 inference mode (args.precision = 'fp32'): the input tile is staged as the unrounded fp32
// rows, every A / B fragment is split in registers and multiplied as 3xTF32 (mma_tf32x3), and the epilogue uses tanhf
// / expf as the reference does.  The weighted sum is fp32 over the fp32 rows in both forms.
template <bool LONG, bool SPLIT>
__global__ void __launch_bounds__(UE_THREADS)
user_encoder_fwd_kernel(const __grid_constant__ UeFwdParams p) {
  extern __shared__ __align__(16) float sm[];
  const int H = p.H, D = p.D, Q = p.Q, DS = D + 4;
  const int HL = LONG ? (H + UE_HMAX - 1) / UE_HMAX * UE_HMAX : UE_HMAX;    // rows of the per-row arrays
  float* sv = sm;                              // [64][D+4]
  float* slog = sv + UE_HMAX * DS;             // [HL]
  float* sz = slog + HL;                       // [HL]
  __shared__ float s_inv;
  const tnr_user_encoder_io io = p.enc[blockIdx.y];
  const int b = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  constexpr int QT = 256;                      // all 32 n-tiles staged (rows >= Q zero-filled): no predicates in the k loop
  float* sW = sz + HL;                         // [2][QT][UE_WS]
  auto load_w = [&](int st, int kc) {
    float* dst = sW + st * QT * UE_WS;
    for (int i = tid; i < QT * (UE_KC / 4); i += UE_THREADS) {
      const int q = i >> 2, c = (i & 3) * 4;
      const bool ok = q < Q;
      cp_async16_zfill(dst + q * UE_WS + c, io.W1 + (size_t)(ok ? q : 0) * D + kc * UE_KC + c, ok);
    }
    cp_async_commit();
  };
  size_t* srow = reinterpret_cast<size_t*>(sW + 2 * QT * UE_WS);     // [HL] row offsets into io.vecs
  for (int h0 = 0; h0 < (LONG ? H : 1); h0 += UE_HMAX) {             // chunk loop (once when !LONG)
  // every stage of the previous chunk was released by the k loop's trailing __syncthreads
  load_w(0, 0);
  // input tile: warp w stages rows w, w + 8, ... (all eight rows of a warp in flight at once), blended if
  // !use_mask and ROUNDED TO TF32 ONCE here (every warp reads every A fragment: converting in the k loop
  // cost 8x the cvt work, and cvt.rna.tf32 is a 3-instruction emulation on sm_100).  The fp32 rows are
  // read again (from L2) for the final weighted sum, so the user vector keeps full fp32 inputs.  SPLIT stages
  // the unrounded fp32 rows: the hi / lo split needs them, and happens per fragment in the k loop.
  {
    const int D4 = D >> 2;
    size_t rows[UE_HMAX / 8];
#pragma unroll
    for (int j = 0; j < UE_HMAX / 8; ++j) {
      const int h = h0 + warp + 8 * j;
      size_t row = (size_t)b * H + (h < H ? h : 0);
      if (p.idx != nullptr) {
        const long long r = p.idx[row];
        row = (r >= 0 && r < p.n_rows) ? (size_t)r : 0;         // unknown id -> row 0 (dataloader.py:74)
      }
      rows[j] = row * D;
      if (lane == 0) srow[h] = rows[j];
    }
    for (int d4 = lane; d4 < D4; d4 += 32) {
      float4 v[UE_HMAX / 8];
#pragma unroll
      for (int j = 0; j < UE_HMAX / 8; ++j)
        v[j] = (h0 + warp + 8 * j < H) ? *reinterpret_cast<const float4*>(io.vecs + rows[j] + d4 * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
      float4 pd = make_float4(0.f, 0.f, 0.f, 0.f);
      if (!p.use_mask) pd = *reinterpret_cast<const float4*>(io.pad_doc + d4 * 4);
#pragma unroll
      for (int j = 0; j < UE_HMAX / 8; ++j) {
        const int h = h0 + warp + 8 * j;
        float4 x = v[j];
        if (!p.use_mask && h < H) {
          const float m = p.mask[(size_t)b * H + h], om = 1.0f - m;
          x.x = x.x * m + pd.x * om; x.y = x.y * m + pd.y * om; x.z = x.z * m + pd.z * om; x.w = x.w * m + pd.w * om;
        }
        if constexpr (SPLIT) {
          *reinterpret_cast<float4*>(sv + (h - h0) * DS + d4 * 4) = x;
        } else {
          uint4 tq = make_uint4(f2tf32(x.x), f2tf32(x.y), f2tf32(x.z), f2tf32(x.w));
          *reinterpret_cast<uint4*>(sv + (h - h0) * DS + d4 * 4) = tq;
        }
      }
    }
  }
  if (tid < UE_HMAX) slog[h0 + tid] = 0.f;
  const int MT = (min(H - h0, UE_HMAX) + 15) >> 4;
  float acc[4][4][4];
#pragma unroll
  for (int mt = 0; mt < 4; ++mt)
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int c = 0; c < 4; ++c) acc[mt][i][c] = 0.f;
  // warp w owns n-tiles w, w+8, w+16, w+24 (Q <= 256)
  const int NK = D / UE_KC;
  for (int kc = 0; kc < NK; ++kc) {
    if (kc + 1 < NK) { load_w((kc + 1) & 1, kc + 1); cp_async_wait<1>(); } else { cp_async_wait<0>(); }
    __syncthreads();                           // chunk kc landed for everyone (first pass: the input tile too)
    const float* w = sW + (kc & 1) * QT * UE_WS;
#pragma unroll
    for (int k8 = 0; k8 < UE_KC / 8; ++k8) {
      if constexpr (SPLIT) {
        uint32_t bh[4][2], bl[4][2];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float* wr = w + ((warp + 8 * i) * 8 + g) * UE_WS + k8 * 8 + t;
          split_tf32(wr[0], bh[i][0], bl[i][0]);
          split_tf32(wr[4], bh[i][1], bl[i][1]);
        }
#pragma unroll
        for (int mt = 0; mt < 4; ++mt) {
          if (mt < MT) {                         // block-uniform
            uint32_t ah[4], al[4];
            const float* r0 = sv + (mt * 16 + g) * DS + kc * UE_KC + k8 * 8 + t;
            split_tf32(r0[0], ah[0], al[0]);
            split_tf32(r0[8 * DS], ah[1], al[1]);
            split_tf32(r0[4], ah[2], al[2]);
            split_tf32(r0[8 * DS + 4], ah[3], al[3]);
#pragma unroll
            for (int i = 0; i < 4; ++i) mma_tf32x3(acc[mt][i], ah, al, bh[i][0], bh[i][1], bl[i][0], bl[i][1]);
          }
        }
      } else {
        uint32_t bf[4][2];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float* wr = w + ((warp + 8 * i) * 8 + g) * UE_WS + k8 * 8 + t;
          bf[i][0] = f2tf32(wr[0]);
          bf[i][1] = f2tf32(wr[4]);
        }
#pragma unroll
        for (int mt = 0; mt < 4; ++mt) {
          if (mt < MT) {                         // block-uniform
            uint32_t a[4];
            const uint32_t* r0 = reinterpret_cast<const uint32_t*>(sv) + (mt * 16 + g) * DS + kc * UE_KC + k8 * 8 + t;
            a[0] = r0[0]; a[1] = r0[8 * DS]; a[2] = r0[4]; a[3] = r0[8 * DS + 4];
#pragma unroll
            for (int i = 0; i < 4; ++i) mma_tf32(acc[mt][i], a, bf[i][0], bf[i][1]);    // n-tiles past Q multiply zeros
          }
        }
      }
    }
    __syncthreads();                           // everyone is done with this stage before it is refilled
  }
  // epilogue: e = tanh(acc + b1); partial logits
  float lp[4][2];
#pragma unroll
  for (int mt = 0; mt < 4; ++mt) { lp[mt][0] = 0.f; lp[mt][1] = 0.f; }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int q = (warp + 8 * i) * 8 + 2 * t + e;
      if (q >= Q) continue;
      const float bq = io.b1[q], wq = io.w2[q];
#pragma unroll
      for (int mt = 0; mt < 4; ++mt) {
        if (mt >= MT) continue;
#pragma unroll
        for (int hi = 0; hi < 2; ++hi) {
          const int h = h0 + mt * 16 + g + hi * 8;
          const float ev = SPLIT ? tanhf(acc[mt][i][hi * 2 + e] + bq) : tanh_exp(acc[mt][i][hi * 2 + e] + bq);
          lp[mt][hi] = fmaf(ev, wq, lp[mt][hi]);
          if (io.e_out != nullptr && h < H) io.e_out[((size_t)b * H + h) * Q + q] = ev;
        }
      }
    }
  }
#pragma unroll
  for (int mt = 0; mt < 4; ++mt)
#pragma unroll
    for (int hi = 0; hi < 2; ++hi) {
      float v = lp[mt][hi];
      v += __shfl_xor_sync(0xffffffffu, v, 1);
      v += __shfl_xor_sync(0xffffffffu, v, 2);
      if (t == 0 && mt < MT) atomicAdd(&slog[h0 + mt * 16 + g + hi * 8], v);
    }
  }                                            // chunk loop
  __syncthreads();
  if constexpr (LONG) {                        // one softmax over all H rows
    __shared__ float s_part[UE_THREADS / 32];
    float s = 0.f;
    for (int h = tid; h < H; h += UE_THREADS) {
      float al = SPLIT ? expf(slog[h] + io.b2[0]) : __expf(slog[h] + io.b2[0]);
      if (p.use_mask) al *= p.mask[(size_t)b * H + h];
      sz[h] = al;
      s += al;
    }
    s = warp_sum(s);
    if (lane == 0) s_part[warp] = s;
    __syncthreads();
    if (warp == 0) {
      s = lane < UE_THREADS / 32 ? s_part[lane] : 0.f;
      s = warp_sum(s);
      if (lane == 0) s_inv = 1.0f / (s + 1e-8f);
    }
    __syncthreads();
    if (io.a_out != nullptr)
      for (int h = tid; h < H; h += UE_THREADS) io.a_out[(size_t)b * H + h] = sz[h] * s_inv;
  } else {
    if (tid < UE_HMAX) {
      float al = 0.f;
      if (tid < H) {
        al = SPLIT ? expf(slog[tid] + io.b2[0]) : __expf(slog[tid] + io.b2[0]);
        if (p.use_mask) al *= p.mask[(size_t)b * H + tid];
      }
      sz[tid] = al;
    }
    __syncthreads();
    if (warp == 0) {
      float s = sz[lane] + sz[lane + 32];
      s = warp_sum(s);
      if (lane == 0) s_inv = 1.0f / (s + 1e-8f);
    }
    __syncthreads();
    if (tid < H && io.a_out != nullptr) io.a_out[(size_t)b * H + tid] = sz[tid] * s_inv;
  }
  const float inv = s_inv;
  for (int d = tid; d < D; d += UE_THREADS) {     // fp32 rows again (L2-hot): sv holds their TF32 roundings
    float u = 0.f;
    const float pd = p.use_mask ? 0.f : io.pad_doc[d];
#pragma unroll 10
    for (int h = 0; h < H; ++h) {
      float x = io.vecs[srow[h] + d];
      if (!p.use_mask) {
        const float m = p.mask[(size_t)b * H + h];
        x = x * m + pd * (1.0f - m);
      }
      u = fmaf(sz[h] * inv, x, u);
    }
    io.user[(size_t)b * D + d] = u;
  }
}

// ----------------------------------------------------------------------------------
// user encoder forward for SCORING (one encoder, thousands of impressions, no e_out): three kernels.
//   (0) ue_compact_kernel: the ids of the history rows with mask != 0 (about half of all (b, h) are front padding).
//   (1) ue_logits_kernel: logit[r] = w2 . tanh(W1 x_r + b1) as ONE flat TF32 GEMM over the live rows on the 5th-gen
//       tensor cores: tcgen05.mma.cta_group::2.kind::tf32, M = 256 rows per CTA PAIR (128 per CTA), N = 208 (Q padded),
//       K = D, fp32 accumulators in TMEM (2 x 256 columns: the epilogue of a tile overlaps the MMAs of the next).
//       W1 is RESIDENT in shared memory for the whole kernel, split over the pair: each CTA holds 104 of the 208 padded
//       output columns for all of K (104 x D x 4 B = 106 KB at D = 256, ONE cp.async.bulk of the pre-swizzled,
//       TF32-rounded image made by ue_pack_w1_kernel) -- cta_group::2 reads the two halves of B from the two SMs, so
//       every history row is fetched from HBM / L2 once, by the CTA that owns it.  The rows are GATHERED by index from
//       the news table (dataloader.py:295 fused): four loader warps per CTA issue 16-byte cp.async copies straight into
//       the 128B-swizzled K-major layout the MMA descriptors read (chunk c of row r lands at r * 128 + ((c ^ (r & 7))
//       << 4) of a 32-float k-block), a 6-stage ring of 16 KB k-blocks that runs on across tiles.  No thread ever waits
//       for its copies: each loader thread posts cp.async.mbarrier.arrive.noinc on the stage's "landed" barrier, which
//       fires when its copies have landed (a wait_group + fence + arrive per stage made the fence wait for EVERY copy
//       in flight -- MEMBAR.ALL.CTA at 13 % of the stall samples, 77 us); the peer CTA's landed barriers are forwarded
//       to the leader by one relay thread (release.cluster), and the next tile's row indices are looked up one tile
//       ahead.  One elected thread of the leader issues the MMAs and multicasts the stage-free /
//       accumulator-ready commits to both CTAs.  Epilogue: a thread owns a row (a TMEM lane), reads its 208
//       accumulators 32 columns at a time (tcgen05.ld.32x32b.x32), applies + b1, tanh, . w2 in registers and writes
//       the logit -- no atomics, no cross-lane reduction.  pad_doc branch: W1 (m v + (1 - m) pad) = m (W1 v) +
//       (1 - m) (W1 pad): the blend is applied to the accumulators with P = W1 pad from the packed image.
//       What this replaced, measured on the 4 096-impression eval step:
//         v1 per-impression kernel, W1 fragments from L2 per k-step ......................... 519 us
//         v3 flat GEMM, 64-row tiles, W1 chunks re-streamed per tile (852 MB of L2 reads) ... 545 us
//         v5 mma.sync TF32, W1 halves resident, live-row list, logit halves by atomicAdd .... 109 us (tensor pipe 36 %)
//   (2) ue_pool_kernel: warp per impression, alpha = exp(logit + b2) [* mask], a = alpha / (sum + 1e-8),
//       user = sum_h a_h x_h over the fp32 rows (gathered again; HBM / L2 bound).
// ----------------------------------------------------------------------------------
constexpr int UL_ROWS = 128;                       // rows per CTA and tile (256 per pair)
constexpr int UL_KB = 32;                          // floats per k-block: 128 B, one swizzle row
constexpr int UL_QT = 208, UL_HALF = UL_QT / 2;    // padded query dim (UMMA N) and the W1 rows one CTA holds
constexpr int UL_STAGES = 6;                       // A ring depth (k-blocks of 16 KB)
constexpr int UL_DMAX = 256;
constexpr int UL_A_BYTES = UL_ROWS * 128;          // one k-block of the A tile: 16 KB
constexpr int UL_W_KB_BYTES = UL_HALF * 128;       // one k-block of a W1 half: 13 KB (13 swizzle atoms)
constexpr int UL_EPI_WARPS = 4, UL_GROUP_WARPS = 4, UL_LOAD_WARPS = 2 * UL_GROUP_WARPS;
constexpr int UL_THREADS = 32 * (UL_EPI_WARPS + 2 + UL_LOAD_WARPS);      // epilogue 0-3, MMA 4, TMEM / W1 5, loaders 6-13
static_assert(UL_STAGES % 2 == 0, "the two loader groups own alternate stages");
constexpr int UL_TMEM_COLS = 512;                  // two accumulator stages of 256 columns (208 used)
constexpr int UL_NBARS = 3 * UL_STAGES + 5;

__host__ __device__ constexpr int ul_smem_bytes(int D) {
  return (D / UL_KB) * UL_W_KB_BYTES + UL_STAGES * UL_A_BYTES + 3 * UL_QT * 4 + UL_NBARS * 8 + 16 + 1024 /*align slack*/;
}
// floats of the packed W1 image: the swizzled halves, then P = W1 pad [208], then c_pad = w2 . tanh(P + b1), padding
__host__ __device__ constexpr long long ul_packed_floats(int D) { return (long long)UL_QT * D + UL_QT + 4; }

struct UlParams {
  const float* vecs;          // [R, D] rows, or the [n_rows, D] table when idx != nullptr
  const int32_t* idx;         // [R] or nullptr
  long long n_rows;
  const float *mask, *W1, *b1, *w2;           // W1: the PACKED image (ue_pack_w1_kernel)
  float* logits;              // [R]; written for the live rows only
  const int32_t* live;        // [n_live] ids of the rows with mask != 0 (ue_compact_kernel; any order)
  const int32_t* n_live;      // device scalar
  int R, D, Q;
#ifdef UL_TIMING
  long long* dbg;             // debug build: clock64 stamps of CTA 0 (tools/ul_timing.py)
#endif
};

// live[] <- the rows r < R with mask[r] != 0, in any order (warp-aggregated atomic append).  Only these go through
// the logits GEMM: at MIND history lengths about half of all (b, h) are front padding.
__global__ void __launch_bounds__(256)
ue_compact_kernel(const float* __restrict__ mask, int R, int32_t* __restrict__ live, int32_t* __restrict__ n_live) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  const bool is_live = r < R && mask[r] != 0.f;
  const unsigned bal = __ballot_sync(0xffffffffu, is_live);
  const int lane = threadIdx.x & 31;
  int base = 0;
  if (lane == 0 && bal) base = atomicAdd(n_live, __popc(bal));
  base = __shfl_sync(0xffffffffu, base, 0);
  if (is_live) live[base + __popc(bal & ((1u << lane) - 1u))] = r;
}

// Packed W1 image.  For CTA half h, k-block kb, row r < 104, 16-byte chunk c < 8, element e < 4 the value
// tf32(W1[h * 104 + r][kb * 32 + c * 4 + e]) (0 past Q) sits at float offset
//   h * 104 * D  +  kb * 104 * 32  +  (r >> 3) * 256  +  (r & 7) * 32  +  ((c ^ (r & 7)) << 2)  +  e :
// exactly the SWIZZLE_128B K-major shared-memory image of the half, so one bulk copy brings it in.  Appended:
// P[q] = sum_d W1[q][d] pad[d] (fp32, from the rounded weights) and c_pad = sum_q w2[q] tanh(P[q] + b1[q]), the logit of
// a history row that IS pad_doc (every masked row of the user_log_mask = False branch, model_bert.py:168-175).
__global__ void ue_pack_w1_kernel(const float* __restrict__ W1, float* __restrict__ Wp, int D, int Q) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= UL_QT * D) return;
  const int q = i / D, d = i - q * D;
  const int h = q / UL_HALF, r = q - h * UL_HALF, kb = d / UL_KB, c = (d % UL_KB) >> 2, e = d & 3;
  float v = 0.f;
  if (q < Q) v = __uint_as_float(f2tf32(W1[(size_t)q * D + d]) & 0xffffe000u);
  Wp[(size_t)h * UL_HALF * D + (size_t)kb * UL_HALF * UL_KB + (r >> 3) * 256 + (r & 7) * 32 + ((c ^ (r & 7)) << 2) + e] = v;
}

__global__ void __launch_bounds__(256)
ue_pack_pad_kernel(const float* __restrict__ W1, const float* __restrict__ pad, const float* __restrict__ b1,
                   const float* __restrict__ w2, float* __restrict__ Wp, int D, int Q) {
  __shared__ float red[8];
  const int q = threadIdx.x;
  float pq = 0.f;
  if (q < Q)
    for (int d = 0; d < D; ++d) pq = fmaf(__uint_as_float(f2tf32(W1[(size_t)q * D + d]) & 0xffffe000u), pad[d], pq);
  float* P = Wp + (size_t)UL_QT * D;
  if (q < UL_QT) P[q] = pq;
  float t = q < Q ? w2[q] * tanh_exp(pq + b1[q]) : 0.f;
  t = warp_sum(t);
  if ((q & 31) == 0) red[q >> 5] = t;
  __syncthreads();
  if (q == 0) {
    float c = 0.f;
    for (int w = 0; w < 8; ++w) c += red[w];
    P[UL_QT] = c;
  }
}

// tanh(x) = 1 - 2 / (1 + 2^(x * 2 log2 e)) on the two MUFU approximations, no range fix-ups (2^y overflows to +inf ->
// rcp gives 0 -> 1; underflows to 0 -> -1): 5 instructions, |error| < 3e-7.  __expf / __fdividef add predicated
// rescaling around each MUFU, and the row epilogue below is MUFU-bound as it is (2 per element, 16 per clock and SM).
__device__ __forceinline__ float tanh_mufu(float x) {
  float r;
  const float e = ex2_approx(x * 2.885390081777927f);
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(1.0f + e));
  return fmaf(-2.0f, r, 1.0f);
}

// NC accumulator columns [c0, c0 + NC) of one row -> sum_c w2[c] tanh(acc[c] (blended) + b1[c]); four independent chains
template <bool BLEND, int NC>
__device__ __forceinline__ float ul_row_chunk(const uint32_t (&r)[32], int c0, const float* __restrict__ sB1,
                                              const float* __restrict__ sW2, const float* __restrict__ sP, float m, float om) {
  float part[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int j = 0; j < NC; j += 4) {
    const float4 b = *reinterpret_cast<const float4*>(sB1 + c0 + j);
    const float4 w = *reinterpret_cast<const float4*>(sW2 + c0 + j);
    const float bb[4] = {b.x, b.y, b.z, b.w}, ww[4] = {w.x, w.y, w.z, w.w};
    float pp[4] = {0.f, 0.f, 0.f, 0.f};
    if (BLEND) {
      const float4 q = *reinterpret_cast<const float4*>(sP + c0 + j);
      pp[0] = q.x; pp[1] = q.y; pp[2] = q.z; pp[3] = q.w;
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      float v = __uint_as_float(r[j + u]);
      if (BLEND) v = fmaf(m, v, om * pp[u]);                   // W1 (m x + (1 - m) pad) = m (W1 x) + (1 - m) (W1 pad)
      part[u] = fmaf(tanh_mufu(v + bb[u]), ww[u], part[u]);
    }
  }
  return (part[0] + part[1]) + (part[2] + part[3]);
}

template <bool BLEND>
__global__ void __launch_bounds__(UL_THREADS, 1)
ue_logits_kernel(const __grid_constant__ UlParams p) {
  using namespace gemm;
  extern __shared__ uint8_t ul_smem_raw[];
  const int D = p.D, Q = p.Q, NKB = D / UL_KB;
  const uint32_t smem_base = (smem_u32(ul_smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = ul_smem_raw + (smem_base - smem_u32(ul_smem_raw));
  // [W1 half: NKB k-blocks of 13 KB][A ring: STAGES x 16 KB][b1 | w2 | P: 3 x 208 floats][barriers][tmem slot]
  const uint32_t sW = smem_base;
  const uint32_t sA = sW + (uint32_t)NKB * UL_W_KB_BYTES;
  float* sVec = reinterpret_cast<float*>(smem_gen + NKB * UL_W_KB_BYTES + UL_STAGES * UL_A_BYTES);
  const uint32_t bar_base = sA + UL_STAGES * UL_A_BYTES + 3 * UL_QT * 4;
  auto landed_bar = [&](int st) { return bar_base + 8u * st; };                      // each CTA: its 128 loader threads' copies
  auto peer_bar = [&](int st) { return bar_base + 8u * (UL_STAGES + st); };           // leader: "the peer's stage landed"
  auto empty_bar = [&](int st) { return bar_base + 8u * (2 * UL_STAGES + st); };      // each CTA: MMA commit (multicast)
  auto tfull_bar = [&](int a) { return bar_base + 8u * (3 * UL_STAGES + a); };        // each CTA: MMA commit (multicast)
  auto tempty_bar = [&](int a) { return bar_base + 8u * (3 * UL_STAGES + 2 + a); };   // leader: both CTAs' epilogue warps
  const uint32_t w_bar = bar_base + 8u * (3 * UL_STAGES + 4);                         // each CTA: its W1 half landed
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem_gen + NKB * UL_W_KB_BYTES + UL_STAGES * UL_A_BYTES +
                                                    3 * UL_QT * 4 + UL_NBARS * 8);
  const int warp = uniform_warp_id(), lane = threadIdx.x & 31;
  const uint32_t cta_rank = cluster_ctarank();                 // 0 = leader of the pair
  const int n_live = *p.n_live;
  const int n_tiles = (n_live + 2 * UL_ROWS - 1) / (2 * UL_ROWS);      // pair tiles of 256 live rows
  const int t_first = (int)(blockIdx.x >> 1), t_stride = (int)(gridDim.x >> 1);

  if (warp == 4 && lane == 0) {
    for (int st = 0; st < UL_STAGES; ++st) {
      mbar_init(landed_bar(st), UL_GROUP_WARPS * 32);
      mbar_init(peer_bar(st), 1);
      mbar_init(empty_bar(st), 1);
    }
    for (int a = 0; a < 2; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), 2 * UL_EPI_WARPS); }
    mbar_init(w_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 5) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "n"(UL_TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  for (int q = threadIdx.x; q < UL_QT; q += UL_THREADS) {
    sVec[q] = q < Q ? p.b1[q] : 0.f;
    sVec[UL_QT + q] = q < Q ? p.w2[q] : 0.f;
    sVec[2 * UL_QT + q] = BLEND ? p.W1[(size_t)UL_QT * D + q] : 0.f;
  }
  tc_fence_before();
  cluster_sync_all();                                          // barriers of both CTAs initialised, TMEM allocated
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 5) {
    // ===================== this CTA's half of W1: one bulk copy of the packed image; the PEER's relay =====================
    if (lane == 0 && t_first < n_tiles) {                      // only a pair with work loads (and later waits for) its W1
      const uint32_t bytes = (uint32_t)NKB * UL_W_KB_BYTES;
      mbar_expect_tx(w_bar, bytes);
      bulk_g2s(sW, p.W1 + (size_t)cta_rank * UL_HALF * D, bytes, w_bar);
      if (cta_rank != 0) {
        // The leader's MMA thread cannot wait on this CTA's barriers: forward "stage landed here" (and, before the
        // first one, "W1 half landed here") to the leader's peer_bar.
        const int my_tiles = (n_tiles - t_first + t_stride - 1) / t_stride;
        const int n_items = my_tiles * NKB;
        const uint32_t peer_remote = mapa_cluster(peer_bar(0), 0);
        mbar_wait(w_bar, 0);
        for (int item = 0; item < n_items; ++item) {
          const int st = item % UL_STAGES;
          mbar_wait(landed_bar(st), ((uint32_t)(item / UL_STAGES)) & 1u);
          fence_proxy_async_smem();                            // cp.async (generic proxy) writes -> the MMA's async-proxy reads
          // relaxed: the data is in THIS SM's shared memory (nothing to publish through the memory hierarchy) and the
          // arrive is control-dependent on the wait above; the release.cluster form costs MEMBAR.ALL.GPU per stage --
          // ~1.5 us on this one thread, i.e. 12 us per tile: it was what the whole pair ran at (62 us)
          mbar_arrive_cluster(peer_remote + 8u * st);
        }
      }
    }
  } else if (warp >= 6) {
    // ===================== loaders: gather this CTA's 128 rows of every tile, k-block by k-block =====================
    // Two groups of four warps take alternate (tile, k-block) items -- group g owns items g, g + 2, ... and, the ring
    // depth being even, stages g, g + 2, g + 4.  One group spent ~750 cycles per stage (free-stage wait, eight copies,
    // arrival, index bookkeeping) against the ~440 the MMAs of a k-block take: the loaders' issue rate, not memory,
    // was the bound once the epilogue was out of the way.
    const int grp = (warp - 6) / UL_GROUP_WARPS;
    const int lt = (threadIdx.x - 6 * 32) & (UL_GROUP_WARPS * 32 - 1);      // 0..127 within the group
    const int piece = lt & 7, rbase = lt >> 3;                 // 16-byte chunk of the k-block row; rows rbase + 16 i
    const uint32_t dst_off = (uint32_t)rbase * 128u + (uint32_t)((piece ^ (rbase & 7)) << 4);    // (r & 7) == (rbase & 7)
    const int my_tiles = t_first < n_tiles ? (n_tiles - t_first + t_stride - 1) / t_stride : 0;
    const int n_items = my_tiles * NKB;
    const float* xsrc[8];
    unsigned xok = 0;
    // The rows of the group's NEXT tile are looked up while this tile streams: live[] ids at its first item, idx[] rows
    // at the second, pointers (+ an L2 prefetch of the whole rows) at the last -- two DEPENDENT index loads per row
    // that would otherwise sit between two tiles.
    int nlive[8];
    long long nrow[8];
    unsigned nok = 0;
    auto look_a = [&](int tl) {                                 // live-list ids of tile tl
      const int r0 = (t_first + tl * t_stride) * (2 * UL_ROWS) + (int)cta_rank * UL_ROWS;
      nok = 0;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int li = r0 + rbase + 16 * i;
        const bool ok = tl < my_tiles && li < n_live;
        nlive[i] = ok ? p.live[li] : 0;
        nok |= (ok ? 1u : 0u) << i;
      }
    };
    auto look_b = [&]() {                                       // table rows
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        long long v = nlive[i];
        if (p.idx != nullptr && ((nok >> i) & 1u)) v = p.idx[nlive[i]];
        nrow[i] = v;
      }
    };
    const float* xnext[8];
    unsigned xok_next = 0;
    auto look_c = [&](bool prefetch) {                          // pointers; unknown id -> row 0 (dataloader.py:74)
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const long long v = nrow[i];
        const size_t src = (p.idx == nullptr || (v >= 0 && v < p.n_rows)) ? (size_t)v : 0;
        xnext[i] = p.vecs + src * D + piece * 4;
        // Pull the WHOLE row towards L2 now, as one burst: the 128-byte k-block slices of a row are copied ~0.5 us
        // apart, i.e. separate DRAM page openings for 1 KB if nothing asks for the row as a unit.  The eight threads
        // that share a row each ask for one of its lines (piece p -> bytes [128 p, 128 p + 128)).
        if (prefetch && ((nok >> i) & 1u) && piece * 32 < D)
          asm volatile("prefetch.global.L2 [%0];" ::"l"(p.vecs + src * D + piece * 32) : "memory");
      }
      xok_next = nok;
    };
    int item = grp;
    int tl = item / NKB, kb = item - tl * NKB;
    int st = grp;                                              // item % UL_STAGES, advanced by 2
    uint32_t phase = 0;
    if (item < n_items) { look_a(tl); look_b(); look_c(true); }
    bool new_tile = true;
    int j = 0, J = 1;                                          // this group's item number within the tile, and how many
    for (; item < n_items; item += 2) {
      if (new_tile) {
#pragma unroll
        for (int i = 0; i < 8; ++i) xsrc[i] = xnext[i];
        xok = xok_next;
        J = (NKB - kb + 1) >> 1;
        j = 0;
        look_a((item + 2 * J) / NKB);                          // the tile this group works on after this one
        new_tile = false;
      }
      if (j == (J > 1 ? 1 : 0)) look_b();
#ifdef UL_TIMING
      if (blockIdx.x == 0 && lt == 0 && item < 64) p.dbg[256 + item * 4 + 0] = clock64();
#endif
      mbar_wait(empty_bar(st), phase ^ 1u);
#ifdef UL_TIMING
      if (blockIdx.x == 0 && lt == 0 && item < 64) p.dbg[256 + item * 4 + 1] = clock64();
#endif
      const uint32_t dst = sA + (uint32_t)st * UL_A_BYTES + dst_off;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const uint32_t sz = ((xok >> i) & 1u) ? 16u : 0u;       // rows past the live list: zero fill
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst + (uint32_t)i * 2048u),
                     "l"(xsrc[i] + kb * UL_KB), "r"(sz) : "memory");
      }
      // this thread's arrival on landed[st] fires when its copies above have landed: nothing here waits for them
      asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(landed_bar(st)) : "memory");
#ifdef UL_TIMING
      if (blockIdx.x == 0 && lt == 0 && item < 64) p.dbg[256 + item * 4 + 2] = clock64();
#endif
      if (j == J - 1) {                                        // last item of the tile for this group
        const int tn = (item + 2) / NKB;                       // == the tile look_a asked about
        look_c(((tn * NKB) & 1) == grp);                       // the group that owns the tile's first k-block prefetches
      }
      ++j;
      kb += 2;
      while (kb >= NKB) { kb -= NKB; ++tl; new_tile = true; }
      st += 2;
      if (st >= UL_STAGES) { st -= UL_STAGES; phase ^= 1u; }
    }
  } else if (warp == 4) {
    // ===================== MMA issuer (the pair leader's elected thread) =====================
    // the whole warp walks the loop and one elected lane issues: operands stay in uniform registers (see gemm_tcgen05.cu)
    if (cta_rank == 0) {
      // D f32, A / B tf32 K-major, N = 208, M = 256 across the pair
      constexpr uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(UL_QT >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
      int item = 0, acc = 0;
      uint32_t acc_phase = 0;
      if (t_first < n_tiles) mbar_wait(w_bar, 0);              // this CTA's W1 half (the peer's comes with its first stage)
      for (int t = t_first; t < n_tiles; t += t_stride) {
        mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
        tc_fence_after();
        const uint32_t tmem_d = __shfl_sync(0xffffffffu, tmem_base, 0) + (uint32_t)(acc * 256);
        for (int kb = 0; kb < NKB; ++kb, ++item) {
          const int st = item % UL_STAGES;
          const uint32_t par = ((uint32_t)(item / UL_STAGES)) & 1u;
          mbar_wait(landed_bar(st), par);                      // this CTA's 128 rows of the k-block
#ifdef UL_TIMING
          if (lane == 0 && blockIdx.x == 0 && item < 64) p.dbg[item * 4 + 0] = clock64();
#endif
          mbar_wait(peer_bar(st), par);                        // the peer's (its data sits in ITS shared memory: no acquire at
                                                               // cluster scope, which costs an L1 invalidate per stage)
#ifdef UL_TIMING
          if (lane == 0 && blockIdx.x == 0 && item < 64) p.dbg[item * 4 + 1] = clock64();
#endif
          fence_proxy_async_smem();
          tc_fence_after();
          const uint64_t adesc = make_desc_kmajor_sw128(sA + (uint32_t)st * UL_A_BYTES);
          const uint64_t bdesc = make_desc_kmajor_sw128(sW + (uint32_t)kb * UL_W_KB_BYTES);
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < UL_KB / 8; ++k)                // kind::tf32: K = 8 per instruction, +32 B inside the atom
              tc_mma_tf32_cta2(tmem_d, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (kb > 0 || k > 0) ? 1u : 0u);
            tc_commit_mc2(empty_bar(st), 3);                   // the stage is free in both CTAs once these MMAs retire
          }
          __syncwarp();
#ifdef UL_TIMING
          if (lane == 0 && blockIdx.x == 0 && item < 64) p.dbg[item * 4 + 2] = clock64();
#endif
        }
        if (elect_one()) tc_commit_mc2(tfull_bar(acc), 3);
        __syncwarp();
        acc ^= 1; if (acc == 0) acc_phase ^= 1u;
      }
    }
  } else {
    // ===================== epilogue: a thread owns a row (TMEM lane) =====================
    const int quarter = warp;                                  // warps 0-3: TMEM lane quarter = warp id % 4
    const float* sB1 = sVec;
    const float* sW2 = sVec + UL_QT;
    const float* sP = sVec + 2 * UL_QT;
    const uint32_t tempty_remote = mapa_cluster(tempty_bar(0), 0);
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int t = t_first; t < n_tiles; t += t_stride) {
      const int li = t * (2 * UL_ROWS) + (int)cta_rank * UL_ROWS + quarter * 32 + lane;
      const int rid = li < n_live ? p.live[li] : -1;
      float m = 1.f, om = 0.f;
      if (BLEND && rid >= 0) { m = p.mask[rid]; om = 1.0f - m; }
#ifdef UL_TIMING
      const int tl_dbg = (t - t_first) / t_stride;
      if (blockIdx.x == 0 && warp == 0 && lane == 0 && tl_dbg < 8) p.dbg[512 + tl_dbg * 4 + 0] = clock64();
#endif
      mbar_wait(tfull_bar(acc), acc_phase);
      tc_fence_after();
#ifdef UL_TIMING
      if (blockIdx.x == 0 && warp == 0 && lane == 0 && tl_dbg < 8) p.dbg[512 + tl_dbg * 4 + 1] = clock64();
#endif
      // 208 columns = six chunks of 32 and one of 16, two register buffers: the next chunk's tcgen05.ld is in flight
      // while this one is evaluated (one load at a time put ~1 000 cycles of TMEM latency in front of every chunk, and
      // a single dependent chain per row made the tile epilogue 15 000 cycles: it, not the loads, set the kernel's time)
      const uint32_t t_row = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * 256);
      uint32_t ra[32], rb[32];
      float logit = 0.f;
      tmem_ld32(t_row, ra);
#pragma unroll
      for (int c0 = 0; c0 < 192; c0 += 64) {
        tmem_ld_wait();
        tmem_ld32(t_row + (uint32_t)(c0 + 32), rb);
        logit += ul_row_chunk<BLEND, 32>(ra, c0, sB1, sW2, sP, m, om);
        tmem_ld_wait();
        tmem_ld32(t_row + (uint32_t)(c0 + 64), ra);            // the last one (c0 + 64 = 192) is the 16-column tail
        logit += ul_row_chunk<BLEND, 32>(rb, c0 + 32, sB1, sW2, sP, m, om);
      }
      tmem_ld_wait();
      logit += ul_row_chunk<BLEND, UL_QT - 192>(ra, 192, sB1, sW2, sP, m, om);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(tempty_remote + 8u * acc);      // this warp is done with the accumulator stage
#ifdef UL_TIMING
      if (blockIdx.x == 0 && warp == 0 && lane == 0 && tl_dbg < 8) p.dbg[512 + tl_dbg * 4 + 2] = clock64();
#endif
      acc ^= 1; if (acc == 0) acc_phase ^= 1u;
      if (rid >= 0) p.logits[rid] = logit;
    }
  }

  tc_fence_before();
  cluster_sync_all();                    // the leader's MMAs also write the peer's TMEM; remote arrives target live CTAs
  if (warp == 5)
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(UL_TMEM_COLS) : "memory");
}

constexpr int UP_WARPS = 4;
// NVT = float4 per lane and row the kernel is compiled for (D <= 128 NVT): D = 256 -> 2, no predicated-off slots.
// The rows with mask != 0 are compacted first (front-padded histories: about half of the H rows), so the streaming
// loop runs over live rows only, eight rows of loads in flight per warp; in the pad_doc branch the masked rows are
// all pad_doc and enter as (sum of their weights) * pad_doc at the end.  HJ = history rows per lane: lane owns rows
// lane + 32 j, j < HJ (HJ = 2 for H <= 64, 16 for H <= 512: 32 KB of static shared memory per block).
template <bool BLEND, int NVT, int HJ>
__global__ void __launch_bounds__(UP_WARPS * 32)
ue_pool_kernel(const float* __restrict__ vecs, const int32_t* __restrict__ idx, long long n_rows,
               const float* __restrict__ mask, const float* __restrict__ pad, const float* __restrict__ b2,
               const float* __restrict__ c_pad, int use_mask, float* __restrict__ logits_a, float* __restrict__ user, int B,
               int H, int D) {
  __shared__ float s_al[UP_WARPS][32 * HJ];             // compacted: weight of live row k
  __shared__ float s_m[UP_WARPS][32 * HJ];              // compacted: its mask value
  __shared__ size_t s_row[UP_WARPS][32 * HJ];           // compacted: its row offset
  const int warp = uniform_warp_id(), lane = threadIdx.x & 31;
  const int b = blockIdx.x * UP_WARPS + warp;
  if (b >= B) return;
  const float bias2 = b2[0];
  float part = 0.f, padw = 0.f;
  float al_own[HJ];                                      // this lane's rows h = lane + 32 j
  int n_live = 0;
#pragma unroll
  for (int j = 0; j < HJ; ++j) {
    const int h = lane + 32 * j;
    float al = 0.f, m = 0.f;
    size_t src = 0;
    const bool in = h < H;
    if (in) {
      const size_t r = (size_t)b * H + h;
      m = mask[r];
      // masked rows never went through the logits GEMM: weight 0 (use_mask) or the pad_doc logit (pad_doc branch)
      al = m != 0.f ? __expf(logits_a[r] + bias2) : (BLEND ? __expf(c_pad[0] + bias2) : 0.f);
      if (use_mask) al *= m;
      src = r;
      if (idx != nullptr) {
        const long long v = idx[r];
        src = (v >= 0 && v < n_rows) ? (size_t)v : 0;
      }
    }
    al_own[j] = al;
    part += al;
    const bool live = in && m != 0.f;
    if (BLEND && in && !live) padw += al;
    const unsigned bal = __ballot_sync(0xffffffffu, live);
    if (live) {
      const int pos = n_live + __popc(bal & ((1u << lane) - 1u));
      s_al[warp][pos] = al;
      s_m[warp][pos] = m;
      s_row[warp][pos] = src * D;
    }
    n_live += __popc(bal);
  }
  part = warp_sum(part);
  padw = warp_sum(padw);
  const float inv = 1.0f / (part + 1e-8f);
  __syncwarp();
#pragma unroll
  for (int j = 0; j < HJ; ++j)
    if (lane + 32 * j < H) logits_a[(size_t)b * H + lane + 32 * j] = al_own[j] * inv;       // a_out
  const int D4 = D >> 2;
  float4 acc[NVT], pd[NVT];
#pragma unroll
  for (int v = 0; v < NVT; ++v) {
    acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);
    pd[v] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (BLEND && v * 32 + lane < D4) pd[v] = *reinterpret_cast<const float4*>(pad + (v * 32 + lane) * 4);
  }
#pragma unroll 8
  for (int k = 0; k < n_live; ++k) {
    const float a = s_al[warp][k] * inv;
    const float* row = vecs + s_row[warp][k];
    const float m = s_m[warp][k], om = 1.0f - m;
#pragma unroll
    for (int v = 0; v < NVT; ++v) {
      if (v * 32 + lane < D4) {
        float4 x = *reinterpret_cast<const float4*>(row + (v * 32 + lane) * 4);
        if (BLEND) {
          x.x = x.x * m + pd[v].x * om; x.y = x.y * m + pd[v].y * om;
          x.z = x.z * m + pd[v].z * om; x.w = x.w * m + pd[v].w * om;
        }
        acc[v].x = fmaf(a, x.x, acc[v].x); acc[v].y = fmaf(a, x.y, acc[v].y);
        acc[v].z = fmaf(a, x.z, acc[v].z); acc[v].w = fmaf(a, x.w, acc[v].w);
      }
    }
  }
  const float pw = padw * inv;
#pragma unroll
  for (int v = 0; v < NVT; ++v)
    if (v * 32 + lane < D4) {
      if (BLEND) {
        acc[v].x = fmaf(pw, pd[v].x, acc[v].x); acc[v].y = fmaf(pw, pd[v].y, acc[v].y);
        acc[v].z = fmaf(pw, pd[v].z, acc[v].z); acc[v].w = fmaf(pw, pd[v].w, acc[v].w);
      }
      *reinterpret_cast<float4*>(user + (size_t)b * D + (v * 32 + lane) * 4) = acc[v];
    }
}

template <bool BLEND, int HJ>
static void ue_pool_launch(int pgrid, cudaStream_t st, const float* vecs, const int32_t* idx, long long n_rows, const float* mask,
                           const float* pad, const float* b2, const float* c_pad, int use_mask, float* a_out, float* user, int B,
                           int H, int D) {
  if (D <= 128) ue_pool_kernel<BLEND, 1, HJ><<<pgrid, UP_WARPS * 32, 0, st>>>(vecs, idx, n_rows, mask, pad, b2, c_pad, use_mask, a_out, user, B, H, D);
  else if (D <= 256) ue_pool_kernel<BLEND, 2, HJ><<<pgrid, UP_WARPS * 32, 0, st>>>(vecs, idx, n_rows, mask, pad, b2, c_pad, use_mask, a_out, user, B, H, D);
  else if (D <= 512) ue_pool_kernel<BLEND, 4, HJ><<<pgrid, UP_WARPS * 32, 0, st>>>(vecs, idx, n_rows, mask, pad, b2, c_pad, use_mask, a_out, user, B, H, D);
  else ue_pool_kernel<BLEND, 8, HJ><<<pgrid, UP_WARPS * 32, 0, st>>>(vecs, idx, n_rows, mask, pad, b2, c_pad, use_mask, a_out, user, B, H, D);
}

template <bool BLEND>
static void ue_pool_launch(int pgrid, cudaStream_t st, const float* vecs, const int32_t* idx, long long n_rows, const float* mask,
                           const float* pad, const float* b2, const float* c_pad, int use_mask, float* a_out, float* user, int B,
                           int H, int D) {
  if (H <= UE_HMAX) ue_pool_launch<BLEND, UE_HMAX / 32>(pgrid, st, vecs, idx, n_rows, mask, pad, b2, c_pad, use_mask, a_out, user, B, H, D);
  else ue_pool_launch<BLEND, UE_HLONG / 32>(pgrid, st, vecs, idx, n_rows, mask, pad, b2, c_pad, use_mask, a_out, user, B, H, D);
}

// ----------------------------------------------------------------------------------
// user encoder backward (student).  d_user [B, D] -> d_vecs (+=) [B*H, D]; dpad / db1 / dw2 / db2
// via fp32 atomics; dU (grad at the fc1 pre-activation) and the blended inputs are written to
// scratch so dW1 += dU^T V runs as one TN GEMM over all impressions afterwards.
// LONG (64 < H <= 512): d alpha needs sum_h a_h (d_user . v_h) over ALL rows first, so the dots are taken straight
// from the fp32 rows (no input tile); then du and the dv product walk the history in 64-row chunks.
// ----------------------------------------------------------------------------------
template <bool LONG>
__global__ void __launch_bounds__(UE_THREADS)
user_encoder_bwd_kernel(const float* __restrict__ vecs, const float* __restrict__ mask, const float* __restrict__ pad_doc,
                        const float* __restrict__ W1, const float* __restrict__ w2, int use_mask,
                        const float* __restrict__ a_in, const float* __restrict__ e_in, const float* __restrict__ d_user,
                        float* __restrict__ d_vecs, float* __restrict__ dpad, float* __restrict__ db1,
                        float* __restrict__ dw2, float* __restrict__ db2, float* __restrict__ dU, float* __restrict__ Vb,
                        int H, int D, int Q) {
  extern __shared__ __align__(16) float sm[];
  const int DS = D + 4, Qp = (Q + 7) & ~7, QS = Qp + 4;
  const int HL = LONG ? (H + UE_HMAX - 1) / UE_HMAX * UE_HMAX : UE_HMAX;
  float* sv = sm;                         // [64][D+4]   blended inputs (!LONG only)
  float* sdu = sv + (LONG ? 0 : UE_HMAX * DS);   // [64][Qp+4]  grad at fc1 pre-activation (rows >= H, cols >= Q zero)
  float* sa = sdu + UE_HMAX * QS;         // [HL]
  float* sdz = sa + HL;                   // [HL]
  float* smk = sdz + HL;                  // [HL]
  float* sdusr = smk + HL;                // [D]
  __shared__ float s_dot;
  const int b = blockIdx.x, tid = threadIdx.x, warp = uniform_warp_id(), lane = tid & 31, g = lane >> 2, t = lane & 3;
  // grid.y column slices: the batch is the grid (32 blocks at the demo shape on 148 SMs), so each impression is cut
  // into S blocks that repeat the cheap part (dz, du) and split the n-tiles of the dv product; slice 0 alone
  // writes dU / Vb and adds the parameter gradients.
  const int slice = blockIdx.y, S = gridDim.y;
  if constexpr (!LONG) {
    // input tile: warp w stages rows w, w + 8, ... with all eight rows of loads in flight (no div / mod per element)
    const int D4 = D >> 2;
    for (int d4 = lane; d4 < D4; d4 += 32) {
      float4 v[UE_HMAX / 8];
#pragma unroll
      for (int j = 0; j < UE_HMAX / 8; ++j) {
        const int h = warp + 8 * j;
        v[j] = h < H ? *reinterpret_cast<const float4*>(vecs + ((size_t)b * H + h) * D + d4 * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
      float4 pd = make_float4(0.f, 0.f, 0.f, 0.f);
      if (!use_mask) pd = *reinterpret_cast<const float4*>(pad_doc + d4 * 4);
#pragma unroll
      for (int j = 0; j < UE_HMAX / 8; ++j) {
        const int h = warp + 8 * j;
        float4 x = v[j];
        if (h < H) {
          if (!use_mask) {
            const float m = mask[(size_t)b * H + h], om = 1.0f - m;
            x.x = x.x * m + pd.x * om; x.y = x.y * m + pd.y * om; x.z = x.z * m + pd.z * om; x.w = x.w * m + pd.w * om;
          }
          if (slice == 0) *reinterpret_cast<float4*>(Vb + ((size_t)b * H + h) * D + d4 * 4) = x;
        }
        *reinterpret_cast<float4*>(sv + h * DS + d4 * 4) = x;
      }
    }
  }
  for (int i = tid; i < UE_HMAX * QS; i += UE_THREADS) sdu[i] = 0.f;
  for (int h = tid; h < HL; h += UE_THREADS) {
    sa[h] = h < H ? a_in[(size_t)b * H + h] : 0.f;
    smk[h] = h < H ? mask[(size_t)b * H + h] : 0.f;
  }
  for (int d = tid; d < D; d += UE_THREADS) sdusr[d] = d_user[(size_t)b * D + d];
  __syncthreads();
  if constexpr (LONG) {
    for (int h = warp; h < H; h += UE_THREADS / 32) {     // da_h = d_user . v_h, straight from the fp32 rows
      const size_t r = ((size_t)b * H + h) * D;
      const float m = smk[h], om = 1.0f - m;
      float s = 0.f;
      for (int d4 = lane; d4 < (D >> 2); d4 += 32) {
        float4 x = *reinterpret_cast<const float4*>(vecs + r + d4 * 4);
        if (!use_mask) {
          const float4 pd = *reinterpret_cast<const float4*>(pad_doc + d4 * 4);
          x.x = x.x * m + pd.x * om; x.y = x.y * m + pd.y * om; x.z = x.z * m + pd.z * om; x.w = x.w * m + pd.w * om;
        }
        if (slice == 0) *reinterpret_cast<float4*>(Vb + r + d4 * 4) = x;
        s = fmaf(sdusr[d4 * 4], x.x, s); s = fmaf(sdusr[d4 * 4 + 1], x.y, s);
        s = fmaf(sdusr[d4 * 4 + 2], x.z, s); s = fmaf(sdusr[d4 * 4 + 3], x.w, s);
      }
      s = warp_sum(s);
      if (lane == 0) sdz[h] = s;
    }
  } else {
    for (int h = warp; h < H; h += UE_THREADS / 32) {       // da_h = d_user . v_h
      float s = 0.f;
      for (int d = lane; d < D; d += 32) s = fmaf(sdusr[d], sv[h * DS + d], s);
      s = warp_sum(s);
      if (lane == 0) sdz[h] = s;
    }
  }
  __syncthreads();
  if (warp == 0) {
    float s = 0.f;
    for (int h = lane; h < H; h += 32) s += sa[h] * sdz[h];
    s = warp_sum(s);
    if (lane == 0) s_dot = s;
  }
  __syncthreads();
  const float dot = s_dot;
  for (int h = tid; h < H; h += UE_THREADS) sdz[h] = sa[h] * (sdz[h] - dot);
  __syncthreads();
  if (warp == 0 && slice == 0) {
    float s = 0.f;
    for (int h = lane; h < H; h += 32) s += sdz[h];
    s = warp_sum(s);
    if (lane == 0) atomicAdd(db2, s);
  }
  for (int h0 = 0; h0 < (LONG ? H : 1); h0 += UE_HMAX) {       // chunk loop (once when !LONG)
    const int HC = LONG ? min(H - h0, UE_HMAX) : H;
    for (int q = tid; q < Q; q += UE_THREADS) {               // du, dw2, db1
      const float w = w2[q];
      float gw2 = 0.f, gb1 = 0.f;
      for (int h = 0; h < HC; ++h) {
        const float ev = e_in[((size_t)b * H + h0 + h) * Q + q];
        const float dz = sdz[h0 + h];
        gw2 = fmaf(dz, ev, gw2);
        const float du = dz * w * (1.0f - ev * ev);
        sdu[h * QS + q] = du;
        if (slice == 0) dU[((size_t)b * H + h0 + h) * Q + q] = du;
        gb1 += du;
      }
      if (slice == 0) {
        atomicAdd(dw2 + q, gw2);
        atomicAdd(db1 + q, gb1);
      }
    }
    __syncthreads();
    // dv[h][d] = a_h dusr_d + sum_q du[h][q] W1[q][d]   (M = 64 rows, N = D, K = Qp), 4 n-tiles per warp per pass.
    // Rows past HC of the last chunk hold the previous chunk's du: their outputs are never stored.
    const int MT = (HC + 15) >> 4;
    for (int pass = 0; pass * 32 < D / 8; ++pass) {
      float acc[4][4][4];
#pragma unroll
      for (int mt = 0; mt < 4; ++mt)
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int c = 0; c < 4; ++c) acc[mt][i][c] = 0.f;
      int ncol[4];
      bool nv[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int tile = pass * 32 + warp + 8 * i;
        ncol[i] = tile * 8;
        nv[i] = ncol[i] < D && ((tile >> 3) % S) == slice;      // groups of 8 n-tiles go round the slices (warp-uniform)
      }
      if (!(nv[0] || nv[1] || nv[2] || nv[3])) continue;
      for (int ks = 0; ks < Qp / 8; ++ks) {
        uint32_t bf[4][2];
        const int q0 = ks * 8 + t;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          bf[i][0] = f2tf32((nv[i] && q0 < Q) ? __ldg(W1 + (size_t)q0 * D + ncol[i] + g) : 0.f);
          bf[i][1] = f2tf32((nv[i] && q0 + 4 < Q) ? __ldg(W1 + (size_t)(q0 + 4) * D + ncol[i] + g) : 0.f);
        }
#pragma unroll
        for (int mt = 0; mt < 4; ++mt) {
          if (mt < MT) {
            uint32_t a[4];
            const float* r0 = sdu + (mt * 16 + g) * QS + ks * 8 + t;
            a[0] = f2tf32(r0[0]); a[1] = f2tf32(r0[8 * QS]); a[2] = f2tf32(r0[4]); a[3] = f2tf32(r0[8 * QS + 4]);
#pragma unroll
            for (int i = 0; i < 4; ++i)
              if (nv[i]) mma_tf32(acc[mt][i], a, bf[i][0], bf[i][1]);
          }
        }
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        if (!nv[i]) continue;
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int d = ncol[i] + 2 * t + e;
          float gpad = 0.f;
#pragma unroll
          for (int mt = 0; mt < 4; ++mt) {
            if (mt >= MT) continue;
#pragma unroll
            for (int hi = 0; hi < 2; ++hi) {
              const int h = mt * 16 + g + hi * 8;
              if (h >= HC) continue;
              const float tv = fmaf(sa[h0 + h], sdusr[d], acc[mt][i][hi * 2 + e]);
              float* dst = d_vecs + ((size_t)b * H + h0 + h) * D + d;
              if (use_mask) {
                *dst += tv;
              } else {
                const float m = smk[h0 + h];
                *dst += tv * m;
                gpad = fmaf(tv, 1.0f - m, gpad);
              }
            }
          }
          if (!use_mask) {
            gpad += __shfl_xor_sync(0xffffffffu, gpad, 4);
            gpad += __shfl_xor_sync(0xffffffffu, gpad, 8);
            gpad += __shfl_xor_sync(0xffffffffu, gpad, 16);
            if (g == 0) atomicAdd(dpad + d, gpad);
          }
        }
      }
    }
    if (LONG) __syncthreads();                 // sdu is rewritten by the next chunk
  }
}

}  // namespace tnr

using namespace tnr;

#define TNR_API extern "C" __attribute__((visibility("default")))

static int launch_sgemm_tn(const float* A, const float* Bm, float* C, float* cbias, int R, int N1, int N2, int batch,
                           long long sA, long long sB, long long sC, long long sbias, cudaStream_t st) {
  TNR_REQUIRE(N1 % 4 == 0 && N2 % 4 == 0, "tnr_sgemm_tn_acc: N1=%d and N2=%d must be multiples of 4", N1, N2);
  TNR_REQUIRE(((uintptr_t)A % 16 == 0) && ((uintptr_t)Bm % 16 == 0) && sA % 4 == 0 && sB % 4 == 0,
              "tnr_sgemm_tn_acc: operands must be 16-byte aligned");
  if (N1 == 0 || N2 == 0 || batch == 0 || R == 0) return 0;
  const int tiles = ((N1 + SG_T - 1) / SG_T) * ((N2 + SG_T - 1) / SG_T) * batch;
  int splits = (2 * num_sms() + tiles - 1) / tiles;
  const int max_splits = (R + 4 * SG_K - 1) / (4 * SG_K);
  if (splits > max_splits) splits = max_splits;
  if (splits < 1) splits = 1;
  int rows_per_split = (R + splits - 1) / splits;
  rows_per_split = (rows_per_split + SG_K - 1) / SG_K * SG_K;
  splits = (R + rows_per_split - 1) / rows_per_split;
  dim3 grid((N2 + SG_T - 1) / SG_T, (N1 + SG_T - 1) / SG_T, batch * splits);
  sgemm_tn_kernel<<<grid, SG_THREADS, 0, st>>>(A, Bm, C, cbias, R, N1, N2, splits, rows_per_split, sA, sB, sC, sbias);
  TNR_LAUNCH_CHECK();
  return 0;
}

template <bool SPLIT>
static int launch_sgemm_nt(const char* who, const float* A, const float* Bm, const float* bias, float* C, int M, int N,
                           int K, int batch, long long sA, long long sB, long long sbias, long long sC, cudaStream_t st) {
  TNR_REQUIRE(K % 4 == 0, "%s: K=%d must be a multiple of 4", who, K);
  TNR_REQUIRE(((uintptr_t)A % 16 == 0) && ((uintptr_t)Bm % 16 == 0) && sA % 4 == 0 && sB % 4 == 0,
              "%s: operands must be 16-byte aligned", who);
  if (M == 0 || N == 0 || batch == 0) return 0;
  dim3 grid((N + SG_T - 1) / SG_T, (M + SG_T - 1) / SG_T, batch);
  sgemm_nt_kernel<SPLIT><<<grid, SG_THREADS, 0, st>>>(A, Bm, bias, C, M, N, K, sA, sB, sbias, sC);
  TNR_LAUNCH_CHECK();
  return 0;
}

TNR_API int tnr_sgemm_nt(const float* A, const float* Bm, const float* bias, float* C, int M, int N, int K, int batch,
                         long long sA, long long sB, long long sbias, long long sC, void* stream) {
  return launch_sgemm_nt<false>("tnr_sgemm_nt", A, Bm, bias, C, M, N, K, batch, sA, sB, sbias, sC,
                                reinterpret_cast<cudaStream_t>(stream));
}

TNR_API int tnr_sgemm_nt_f32(const float* A, const float* Bm, const float* bias, float* C, int M, int N, int K, int batch,
                             long long sA, long long sB, long long sbias, long long sC, void* stream) {
  return launch_sgemm_nt<true>("tnr_sgemm_nt_f32", A, Bm, bias, C, M, N, K, batch, sA, sB, sbias, sC,
                               reinterpret_cast<cudaStream_t>(stream));
}

TNR_API int tnr_sgemm_tn_acc(const float* A, const float* Bm, float* C, float* cbias, int R, int N1, int N2, int batch,
                             long long sA, long long sB, long long sC, long long sbias, void* stream) {
  return launch_sgemm_tn(A, Bm, C, cbias, R, N1, N2, batch, sA, sB, sC, sbias, reinterpret_cast<cudaStream_t>(stream));
}

static int ue_check(const char* who, int H, int D, int Q) {
  TNR_REQUIRE(H >= 1 && H <= UE_HLONG, "%s: history length %d not supported (1..%d)", who, H, UE_HLONG);
  TNR_REQUIRE(D % 8 == 0 && D >= 8 && D <= 768, "%s: D=%d must be a multiple of 8 in 8..768", who, D);
  TNR_REQUIRE(Q >= 1 && Q <= 256, "%s: query dim %d not supported (1..256)", who, Q);
  return 0;
}

template <bool SPLIT>
static int ue_fwd_launch(const tnr_user_encoder_io* enc, int n_enc, const float* mask, const int32_t* idx, long long n_rows,
                         int use_mask, int B, int H, int D, int Q, cudaStream_t st) {
  if (ue_check("tnr_user_encoder_fwd", H, D, Q)) return 1;
  TNR_REQUIRE(D % UE_KC == 0, "tnr_user_encoder_fwd: D=%d must be a multiple of %d", D, UE_KC);
  TNR_REQUIRE(n_enc >= 1 && n_enc <= UE_MAX_ENC, "tnr_user_encoder_fwd_multi: n_enc=%d out of range (1..%d)", n_enc, UE_MAX_ENC);
  if (B == 0) return 0;
  UeFwdParams p;
  for (int i = 0; i < n_enc; ++i) p.enc[i] = enc[i];
  for (int i = n_enc; i < UE_MAX_ENC; ++i) p.enc[i] = enc[0];
  p.mask = mask; p.idx = idx; p.n_rows = n_rows; p.use_mask = use_mask; p.H = H; p.D = D; p.Q = Q;
  if (H <= UE_HMAX) {
    const int smem = (UE_HMAX * (D + 4) + 2 * UE_HMAX + 2 * 256 * UE_WS) * 4 + UE_HMAX * 8;
    TNR_SET_SMEM((user_encoder_fwd_kernel<false, SPLIT>), smem);
    user_encoder_fwd_kernel<false, SPLIT><<<dim3(B, n_enc), UE_THREADS, smem, st>>>(p);
  } else {
    const int HL = (H + UE_HMAX - 1) / UE_HMAX * UE_HMAX;
    const int smem = (UE_HMAX * (D + 4) + 2 * HL + 2 * 256 * UE_WS) * 4 + HL * 8;
    TNR_SET_SMEM((user_encoder_fwd_kernel<true, SPLIT>), smem);
    user_encoder_fwd_kernel<true, SPLIT><<<dim3(B, n_enc), UE_THREADS, smem, st>>>(p);
  }
  TNR_LAUNCH_CHECK();
  return 0;
}

TNR_API int tnr_user_encoder_fwd_multi(const tnr_user_encoder_io* enc, int n_enc, const float* mask, int use_mask, int B,
                                       int H, int D, int Q, void* stream) {
  return ue_fwd_launch<false>(enc, n_enc, mask, nullptr, 0, use_mask, B, H, D, Q, reinterpret_cast<cudaStream_t>(stream));
}

template <bool SPLIT>
static int ue_fwd_gather(const char* who, const float* table, long long n_rows, const int32_t* idx, const float* mask,
                         const float* pad_doc, const float* W1, const float* b1, const float* w2, const float* b2,
                         int use_mask, float* user, float* a_out, int B, int H, int D, int Q, void* stream) {
  TNR_REQUIRE(idx != nullptr && n_rows >= 1, "%s: idx and a non-empty table are required", who);
  tnr_user_encoder_io io;
  io.vecs = table; io.pad_doc = pad_doc; io.W1 = W1; io.b1 = b1; io.w2 = w2; io.b2 = b2;
  io.user = user; io.a_out = a_out; io.e_out = nullptr;
  return ue_fwd_launch<SPLIT>(&io, 1, mask, idx, n_rows, use_mask, B, H, D, Q, reinterpret_cast<cudaStream_t>(stream));
}

TNR_API int tnr_user_encoder_fwd_gather(const float* table, long long n_rows, const int32_t* idx, const float* mask,
                                        const float* pad_doc, const float* W1, const float* b1, const float* w2,
                                        const float* b2, int use_mask, float* user, float* a_out, int B, int H, int D,
                                        int Q, void* stream) {
  return ue_fwd_gather<false>("tnr_user_encoder_fwd_gather", table, n_rows, idx, mask, pad_doc, W1, b1, w2, b2, use_mask,
                              user, a_out, B, H, D, Q, stream);
}

TNR_API int tnr_user_encoder_fwd_gather_f32(const float* table, long long n_rows, const int32_t* idx, const float* mask,
                                            const float* pad_doc, const float* W1, const float* b1, const float* w2,
                                            const float* b2, int use_mask, float* user, float* a_out, int B, int H, int D,
                                            int Q, void* stream) {
  return ue_fwd_gather<true>("tnr_user_encoder_fwd_gather_f32", table, n_rows, idx, mask, pad_doc, W1, b1, w2, b2,
                             use_mask, user, a_out, B, H, D, Q, stream);
}

TNR_API int tnr_user_encoder_fwd(const float* vecs, const float* mask, const float* pad_doc, const float* W1,
                                 const float* b1, const float* w2, const float* b2, int use_mask, float* user,
                                 float* a_out, float* e_out, int B, int H, int D, int Q, void* stream) {
  tnr_user_encoder_io io;
  io.vecs = vecs; io.pad_doc = pad_doc; io.W1 = W1; io.b1 = b1; io.w2 = w2; io.b2 = b2;
  io.user = user; io.a_out = a_out; io.e_out = e_out;
  return tnr_user_encoder_fwd_multi(&io, 1, mask, use_mask, B, H, D, Q, stream);
}

TNR_API int tnr_user_encoder_fwd_f32(const float* vecs, const float* mask, const float* pad_doc, const float* W1,
                                     const float* b1, const float* w2, const float* b2, int use_mask, float* user,
                                     float* a_out, float* e_out, int B, int H, int D, int Q, void* stream) {
  tnr_user_encoder_io io;
  io.vecs = vecs; io.pad_doc = pad_doc; io.W1 = W1; io.b1 = b1; io.w2 = w2; io.b2 = b2;
  io.user = user; io.a_out = a_out; io.e_out = e_out;
  return ue_fwd_launch<true>(&io, 1, mask, nullptr, 0, use_mask, B, H, D, Q, reinterpret_cast<cudaStream_t>(stream));
}

// ---- scoring path: flat logits GEMM + per-impression pooling (see ue_logits_kernel) -------------------
static int ue_score_check(const char* who, int H, int D, int Q) {
  TNR_REQUIRE(H >= 1 && H <= UE_HLONG, "%s: history length %d not supported (1..%d)", who, H, UE_HLONG);
  TNR_REQUIRE(D % UL_KB == 0 && D >= UL_KB && D <= UL_DMAX, "%s: D=%d must be a multiple of %d in %d..%d", who, D, UL_KB, UL_KB, UL_DMAX);
  TNR_REQUIRE(Q >= 1 && Q <= UL_QT, "%s: query dim %d not supported (1..%d)", who, Q, UL_QT);
  return 0;
}

TNR_API long long tnr_user_encoder_packed_w1_floats(int D) { return ul_packed_floats(D); }

TNR_API int tnr_user_encoder_pack_w1(const float* W1, const float* pad_doc, const float* b1, const float* w2, float* packed,
                                     int D, int Q, void* stream) {
  if (ue_score_check("tnr_user_encoder_pack_w1", 1, D, Q)) return 1;
  TNR_REQUIRE((uintptr_t)packed % 16 == 0, "tnr_user_encoder_pack_w1: packed must be 16-byte aligned");
  TNR_REQUIRE(W1 != nullptr && pad_doc != nullptr && b1 != nullptr && w2 != nullptr, "tnr_user_encoder_pack_w1: null parameter");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int total = UL_QT * D;
  ue_pack_w1_kernel<<<(total + 255) / 256, 256, 0, st>>>(W1, packed, D, Q);
  TNR_LAUNCH_CHECK();
  ue_pack_pad_kernel<<<1, 256, 0, st>>>(W1, pad_doc, b1, w2, packed, D, Q);
  TNR_LAUNCH_CHECK();
  return 0;
}

#ifdef UL_TIMING
TNR_API long long tnr_user_encoder_score_ws_bytes(int B, int H) { return ((long long)B * H + 4) * 4 + 8192; }
#else
TNR_API long long tnr_user_encoder_score_ws_bytes(int B, int H) { return ((long long)B * H + 4) * 4; }
#endif

template <bool BLEND>
static int ue_logits_launch(const UlParams& p, int pairs, int smem, cudaStream_t st) {
  TNR_SET_SMEM(ue_logits_kernel<BLEND>, ul_smem_bytes(UL_DMAX));
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2 * pairs);
  cfg.blockDim = dim3(UL_THREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  TNR_CHECK_CUDA(cudaLaunchKernelEx(&cfg, ue_logits_kernel<BLEND>, p));
  return 0;
}

TNR_API int tnr_user_encoder_score(const float* vecs, long long n_rows, const int32_t* idx, const float* mask,
                                   const float* pad_doc, const float* w1_packed, const float* b1, const float* w2,
                                   const float* b2, int use_mask, float* user, float* a_out, void* workspace, int B, int H,
                                   int D, int Q, void* stream) {
  if (ue_score_check("tnr_user_encoder_score", H, D, Q)) return 1;
  TNR_REQUIRE(a_out != nullptr && user != nullptr && w1_packed != nullptr && (uintptr_t)w1_packed % 16 == 0,
              "tnr_user_encoder_score: a_out [B,H] (logits workspace), user and a 16-byte aligned packed W1 are required");
  TNR_REQUIRE(workspace != nullptr && (uintptr_t)workspace % 16 == 0,
              "tnr_user_encoder_score: workspace of tnr_user_encoder_score_ws_bytes(B, H) bytes required");
  TNR_REQUIRE(idx == nullptr || n_rows >= 1, "tnr_user_encoder_score: empty table");
  TNR_REQUIRE((uintptr_t)vecs % 16 == 0, "tnr_user_encoder_score: rows must be 16-byte aligned");
  if (B == 0) return 0;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int R = B * H;
  // workspace: [0] n_live (int32), [4 ..] the live row list
  int32_t* wsi = reinterpret_cast<int32_t*>(workspace);
  TNR_CHECK_CUDA(cudaMemsetAsync(wsi, 0, 16, st));
  ue_compact_kernel<<<(R + 255) / 256, 256, 0, st>>>(mask, R, wsi + 4, wsi);
  TNR_LAUNCH_CHECK();
  UlParams p;
  p.vecs = vecs; p.idx = idx; p.n_rows = n_rows; p.mask = mask; p.W1 = w1_packed; p.b1 = b1; p.w2 = w2;
  p.logits = a_out; p.live = wsi + 4; p.n_live = wsi;
  p.R = R; p.D = D; p.Q = Q;
#ifdef UL_TIMING
  p.dbg = reinterpret_cast<long long*>(reinterpret_cast<char*>(workspace) + ((size_t)R + 4) * 4);
#endif
  const int smem = ul_smem_bytes(D);
  const int n_tiles = (R + 2 * UL_ROWS - 1) / (2 * UL_ROWS);      // upper bound: the live count is only known on the device
  const int pairs = n_tiles < num_sms() / 2 ? n_tiles : num_sms() / 2;
  const int pgrid = (B + UP_WARPS - 1) / UP_WARPS;
  const float* c_pad = w1_packed + (size_t)UL_QT * D + UL_QT;    // logit of a pad_doc row (ue_pack_pad_kernel)
  if (use_mask) {
    if (ue_logits_launch<false>(p, pairs, smem, st)) return 2;
    ue_pool_launch<false>(pgrid, st, vecs, idx, n_rows, mask, pad_doc, b2, c_pad, 1, a_out, user, B, H, D);
  } else {
    if (ue_logits_launch<true>(p, pairs, smem, st)) return 2;
    ue_pool_launch<true>(pgrid, st, vecs, idx, n_rows, mask, pad_doc, b2, c_pad, 0, a_out, user, B, H, D);
  }
  TNR_LAUNCH_CHECK();
  return 0;
}

TNR_API int tnr_user_encoder_bwd(const float* vecs, const float* mask, const float* pad_doc, const float* W1,
                                 const float* w2, int use_mask, const float* a_in, const float* e_in,
                                 const float* d_user, float* d_vecs, float* dpad, float* dW1, float* db1, float* dw2,
                                 float* db2, float* scratch, int B, int H, int D, int Q, void* stream) {
  if (ue_check("tnr_user_encoder_bwd", H, D, Q)) return 1;
  TNR_REQUIRE(Q % 4 == 0, "tnr_user_encoder_bwd: query dim %d must be a multiple of 4", Q);
  TNR_REQUIRE(D <= 512, "tnr_user_encoder_bwd: D=%d too large for shared memory (<= 512)", D);
  TNR_REQUIRE(scratch != nullptr && (uintptr_t)scratch % 16 == 0, "tnr_user_encoder_bwd: scratch [B*H*(Q+D)] fp32 required");
  if (B == 0) return 0;
  const int Qp = (Q + 7) & ~7;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  float* dU = scratch;
  float* Vb = scratch + (size_t)B * H * Q;
  int slices = (2 * num_sms()) / (B > 0 ? B : 1);              // fill the machine: 4 column slices at batch 32
  slices = slices < 1 ? 1 : (slices > 4 ? 4 : slices);
  if (H <= UE_HMAX) {
    const int smem = (UE_HMAX * (D + 4) + UE_HMAX * (Qp + 4) + 3 * UE_HMAX + D) * 4;
    TNR_SET_SMEM(user_encoder_bwd_kernel<false>, smem);
    user_encoder_bwd_kernel<false><<<dim3(B, slices), UE_THREADS, smem, st>>>(vecs, mask, pad_doc, W1, w2, use_mask, a_in, e_in, d_user,
                                                                     d_vecs, dpad, db1, dw2, db2, dU, Vb, H, D, Q);
  } else {
    const int HL = (H + UE_HMAX - 1) / UE_HMAX * UE_HMAX;
    const int smem = (UE_HMAX * (Qp + 4) + 3 * HL + D) * 4;
    TNR_SET_SMEM(user_encoder_bwd_kernel<true>, smem);
    user_encoder_bwd_kernel<true><<<dim3(B, slices), UE_THREADS, smem, st>>>(vecs, mask, pad_doc, W1, w2, use_mask, a_in, e_in, d_user,
                                                                    d_vecs, dpad, db1, dw2, db2, dU, Vb, H, D, Q);
  }
  TNR_LAUNCH_CHECK();
  return launch_sgemm_tn(dU, Vb, dW1, nullptr, B * H, Q, D, 1, 0, 0, 0, 0, st);
}
