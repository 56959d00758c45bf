// fp32 inference path of the news encoder (the 1e-4 parity mode): fp32 activations end to end.
// The contractions run on the bf16 tcgen05 GEMM with each fp32 operand split into two bf16 parts,
// x = hi + lo (hi = bf16_rn(x), lo = bf16_rn(x - hi)), laid out along K so that one GEMM with K' = 3K
// computes A_hi W_hi + A_lo W_hi + A_hi W_lo (the dropped lo * lo term is ~2^-16 relative).
// Everything between the GEMMs (embedding + LayerNorm, residual add + LayerNorm, attention, word pooling)
// is plain fp32 with exact transcendental functions (erfcf for the GELU, expf, tanhf).
#include "common.cuh"

namespace tnr {

// ---- fp32 -> bf16 [hi|lo|hi] (activations) or [hi|hi|lo] (weights), optionally through the exact erf-GELU
// 0.5 v (1 + erf(v / sqrt 2)) written with erfc, which keeps the negative tail (where 1 + erf cancels) accurate to a few
// ulps (the GEMM epilogue's quintic is 2.6e-5 off: too coarse for this mode)
__device__ __forceinline__ float gelu_exact(float v) { return 0.5f * v * erfcf(v * -0.70710678118654752f); }

__device__ __forceinline__ void split1(float v, __nv_bfloat16& hi, __nv_bfloat16& lo) {
  hi = __float2bfloat16_rn(v);
  lo = __float2bfloat16_rn(v - __bfloat162float(hi));
}

template <bool GELU>
__global__ void __launch_bounds__(256)
split_bf16x3_kernel(const float* __restrict__ x, long long rows, int K, int ldx, int weight_layout,
                    __nv_bfloat16* __restrict__ out) {
  const long long total = rows * K;
  const long long K3 = 3LL * K;
  const int off_lo = weight_layout ? 2 * K : K, off_hi2 = weight_layout ? K : 2 * K;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / K;
    const int c = (int)(i - r * K);
    float v = x[r * ldx + c];
    if (GELU) v = gelu_exact(v);
    __nv_bfloat16 hi, lo;
    split1(v, hi, lo);
    __nv_bfloat16* o = out + r * K3 + c;
    o[0] = hi;
    o[off_lo] = lo;
    o[off_hi2] = hi;
  }
}

// 4 columns per thread (K % 4 == 0, ldx % 4 == 0, 16-byte aligned input): one float4 load, three 8-byte stores
template <bool GELU>
__global__ void __launch_bounds__(256)
split_bf16x3_vec4_kernel(const float* __restrict__ x, long long rows, int K, int ldx, int weight_layout,
                         __nv_bfloat16* __restrict__ out) {
  const int K4 = K >> 2;
  const long long total = rows * K4;
  const long long K3 = 3LL * K;
  const int off_lo = weight_layout ? 2 * K : K, off_hi2 = weight_layout ? K : 2 * K;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / K4;
    const int c = (int)(i - r * K4) * 4;
    float4 v = *reinterpret_cast<const float4*>(x + r * ldx + c);
    if (GELU) { v.x = gelu_exact(v.x); v.y = gelu_exact(v.y); v.z = gelu_exact(v.z); v.w = gelu_exact(v.w); }
    __nv_bfloat16 h[4], l[4];
    split1(v.x, h[0], l[0]); split1(v.y, h[1], l[1]); split1(v.z, h[2], l[2]); split1(v.w, h[3], l[3]);
    uint2 hv, lv;
    hv.x = (uint32_t)__bfloat16_as_ushort(h[0]) | ((uint32_t)__bfloat16_as_ushort(h[1]) << 16);
    hv.y = (uint32_t)__bfloat16_as_ushort(h[2]) | ((uint32_t)__bfloat16_as_ushort(h[3]) << 16);
    lv.x = (uint32_t)__bfloat16_as_ushort(l[0]) | ((uint32_t)__bfloat16_as_ushort(l[1]) << 16);
    lv.y = (uint32_t)__bfloat16_as_ushort(l[2]) | ((uint32_t)__bfloat16_as_ushort(l[3]) << 16);
    __nv_bfloat16* o = out + r * K3 + c;
    *reinterpret_cast<uint2*>(o) = hv;
    *reinterpret_cast<uint2*>(o + off_lo) = lv;
    *reinterpret_cast<uint2*>(o + off_hi2) = hv;
  }
}

// ---- row kernels: one warp per row of E = VPL * 256 fp32 values, 8 per lane as two float4 per vector.
// Statistics in two passes (mean, then the centred variance), as torch's LayerNorm does.
constexpr int F32_ROW_WARPS = 8;

template <int VPL>
__device__ __forceinline__ void ln_row_store(float (&x)[VPL * 8], const float* __restrict__ gamma,
                                             const float* __restrict__ beta, float eps, float* __restrict__ y, int lane) {
  constexpr int E = VPL * 256;
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < VPL * 8; ++i) s += x[i];
  const float mean = warp_sum(s) * (1.0f / E);
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < VPL * 8; ++i) { const float d = x[i] - mean; q = fmaf(d, d, q); }
  const float rstd = 1.0f / sqrtf(warp_sum(q) * (1.0f / E) + eps);
#pragma unroll
  for (int v = 0; v < VPL; ++v)
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int col = (v * 32 + lane) * 8 + 4 * h;
      const float4 g = *reinterpret_cast<const float4*>(gamma + col);
      const float4 b = *reinterpret_cast<const float4*>(beta + col);
      const float* xv = x + v * 8 + 4 * h;
      float4 o;
      o.x = (xv[0] - mean) * rstd * g.x + b.x;
      o.y = (xv[1] - mean) * rstd * g.y + b.y;
      o.z = (xv[2] - mean) * rstd * g.z + b.z;
      o.w = (xv[3] - mean) * rstd * g.w + b.w;
      *reinterpret_cast<float4*>(y + col) = o;
    }
}

template <int VPL>
__device__ __forceinline__ void load_row8(float (&x)[VPL * 8], const float* __restrict__ src, int lane) {
#pragma unroll
  for (int v = 0; v < VPL; ++v)
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const float4 a = *reinterpret_cast<const float4*>(src + (v * 32 + lane) * 8 + 4 * h);
      x[v * 8 + 4 * h] = a.x; x[v * 8 + 4 * h + 1] = a.y; x[v * 8 + 4 * h + 2] = a.z; x[v * 8 + 4 * h + 3] = a.w;
    }
}

// out[t] = LN(word[id[t]] + pos[t % L] + type0), ids clamped to [0, vocab) like the bf16 kernel
template <int VPL>
__global__ void __launch_bounds__(F32_ROW_WARPS * 32)
embed_ln_f32_kernel(const int64_t* __restrict__ ids, int ids_ld, int L, long long T, int vocab,
                    const float* __restrict__ word, const float* __restrict__ pos, const float* __restrict__ type0,
                    const float* __restrict__ gamma, const float* __restrict__ beta, float eps, float* __restrict__ out) {
  constexpr int E = VPL * 256;
  const int lane = threadIdx.x & 31;
  const long long t = blockIdx.x * (long long)F32_ROW_WARPS + uniform_warp_id();
  if (t >= T) return;
  const long long n = t / L;
  const int l = (int)(t - n * L);
  long long id = ids[n * ids_ld + l];
  id = id < 0 ? 0 : (id >= vocab ? vocab - 1 : id);
  float x[VPL * 8], p[VPL * 8], ty[VPL * 8];
  load_row8<VPL>(x, word + id * E, lane);
  load_row8<VPL>(p, pos + (size_t)l * E, lane);
  load_row8<VPL>(ty, type0, lane);
#pragma unroll
  for (int i = 0; i < VPL * 8; ++i) x[i] = (x[i] + p[i]) + ty[i];      // the reference's order, modeling.py:168-176
  ln_row_store<VPL>(x, gamma, beta, eps, out + t * E, lane);
}

// y = LN(x + residual)
template <int VPL>
__global__ void __launch_bounds__(F32_ROW_WARPS * 32)
add_ln_f32_kernel(const float* __restrict__ x, const float* __restrict__ res, long long rows, const float* __restrict__ gamma,
                  const float* __restrict__ beta, float eps, float* __restrict__ y) {
  constexpr int E = VPL * 256;
  const int lane = threadIdx.x & 31;
  const long long r = blockIdx.x * (long long)F32_ROW_WARPS + uniform_warp_id();
  if (r >= rows) return;
  float a[VPL * 8], b[VPL * 8];
  load_row8<VPL>(a, x + r * E, lane);
  load_row8<VPL>(b, res + r * E, lane);
#pragma unroll
  for (int i = 0; i < VPL * 8; ++i) a[i] += b[i];
  ln_row_store<VPL>(a, gamma, beta, eps, y + r * E, lane);
}

// ---- attention: ctx = softmax(q k^T / 8 + (1 - mask) * -10000 + relbias[h][j - i]) v, head dim 64, fp32 FFMA.
// Block = (32 queries, head, news), 4 warps of 8 queries; keys stream through shared memory in chunks of 64 with an
// online softmax.  Every key is visited, masked or not: a row whose keys are all padding gets the reference's softmax
// over the -10000-shifted scores, not a zero row.
constexpr int ATF_Q = 32, ATF_KC = 64, ATF_WARPS = 4, ATF_QPW = ATF_Q / ATF_WARPS;

__global__ void __launch_bounds__(ATF_WARPS * 32)
attn_f32_kernel(const float* __restrict__ qkv, const int64_t* __restrict__ mask, int mask_ld,
                const float* __restrict__ relbias, float* __restrict__ ctx, int L, int E) {
  __shared__ __align__(16) float sq[ATF_Q][64];
  __shared__ float sk[ATF_KC][65];
  __shared__ __align__(16) float sv[ATF_KC][64];
  __shared__ float sadd[ATF_KC];
  const int warp = uniform_warp_id(), lane = threadIdx.x & 31;
  const int i0 = blockIdx.x * ATF_Q, h = blockIdx.y;
  const long long n = blockIdx.z;
  const long long row0 = n * L;
  const size_t ld = 3 * (size_t)E;
  const float* rb = relbias + (size_t)h * (2 * L - 1) + (L - 1);       // rb[j - i]
  for (int e = threadIdx.x; e < ATF_Q * 16; e += blockDim.x) {
    const int r = e >> 4, c = (e & 15) * 4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (i0 + r < L) v = *reinterpret_cast<const float4*>(qkv + (row0 + i0 + r) * ld + h * 64 + c);
    *reinterpret_cast<float4*>(&sq[r][c]) = v;
  }
  float m[ATF_QPW], l[ATF_QPW], acc0[ATF_QPW], acc1[ATF_QPW];
#pragma unroll
  for (int r = 0; r < ATF_QPW; ++r) { m[r] = -INFINITY; l[r] = 0.f; acc0[r] = 0.f; acc1[r] = 0.f; }
  for (int kc = 0; kc < L; kc += ATF_KC) {
    const int nk = min(ATF_KC, L - kc);
    __syncthreads();
    for (int e = threadIdx.x; e < ATF_KC * 16; e += blockDim.x) {
      const int r = e >> 4, c = (e & 15) * 4;
      float4 kv = make_float4(0.f, 0.f, 0.f, 0.f), vv = kv;
      if (r < nk) {
        const float* src = qkv + (row0 + kc + r) * ld + h * 64 + c;
        kv = *reinterpret_cast<const float4*>(src + E);
        vv = *reinterpret_cast<const float4*>(src + 2 * E);
      }
      sk[r][c] = kv.x; sk[r][c + 1] = kv.y; sk[r][c + 2] = kv.z; sk[r][c + 3] = kv.w;
      *reinterpret_cast<float4*>(&sv[r][c]) = vv;
    }
    if (threadIdx.x < nk) sadd[threadIdx.x] = (1.0f - (float)mask[n * mask_ld + kc + threadIdx.x]) * -10000.0f;
    __syncthreads();
#pragma unroll
    for (int r = 0; r < ATF_QPW; ++r) {
      const int qr = warp * ATF_QPW + r, qi = i0 + qr;
      if (qi >= L) break;
      float a0 = 0.f, a1 = 0.f;
#pragma unroll 16
      for (int d = 0; d < 64; ++d) {
        const float qd = sq[qr][d];
        a0 = fmaf(qd, sk[lane][d], a0);
        a1 = fmaf(qd, sk[lane + 32][d], a1);
      }
      const float s0 = lane < nk ? (a0 * 0.125f + sadd[lane]) + rb[kc + lane - qi] : -INFINITY;
      const float s1 = lane + 32 < nk ? (a1 * 0.125f + sadd[lane + 32]) + rb[kc + lane + 32 - qi] : -INFINITY;
      const float mnew = fmaxf(m[r], warp_max(fmaxf(s0, s1)));
      const float corr = expf(m[r] - mnew);
      const float p0 = expf(s0 - mnew), p1 = expf(s1 - mnew);
      l[r] = l[r] * corr + warp_sum(p0 + p1);
      float c0 = acc0[r] * corr, c1 = acc1[r] * corr;
      for (int j = 0; j < nk; ++j) {
        const float pj = __shfl_sync(0xffffffffu, j < 32 ? p0 : p1, j & 31);
        c0 = fmaf(pj, sv[j][lane], c0);
        c1 = fmaf(pj, sv[j][lane + 32], c1);
      }
      acc0[r] = c0; acc1[r] = c1;
      m[r] = mnew;
    }
  }
#pragma unroll
  for (int r = 0; r < ATF_QPW; ++r) {
    const int qi = i0 + warp * ATF_QPW + r;
    if (qi >= L) break;
    float* o = ctx + (row0 + qi) * (size_t)E + h * 64;
    o[lane] = acc0[r] / l[r];
    o[lane + 32] = acc1[r] / l[r];
  }
}

// ---- word pooling: a_s = exp(tanh(u_s) . w2 + b2) / (sum_s + 1e-8) (no max subtraction, model_bert.py:15-34);
// out[n] = sum_s a_s x[n, s].  One block per news row.
constexpr int POOLF_THREADS = 256;

__global__ void __launch_bounds__(POOLF_THREADS)
attnpool_f32_kernel(const float* __restrict__ x, const float* __restrict__ u, int ldq, int Q, const float* __restrict__ w2,
                    const float* __restrict__ b2, float* __restrict__ out, int S, int C) {
  extern __shared__ float pa[];          // S weights, then the normaliser
  const int warp = uniform_warp_id(), lane = threadIdx.x & 31;
  const long long n = blockIdx.x;
  for (int s = warp; s < S; s += POOLF_THREADS / 32) {
    const float* row = u + (n * S + s) * (size_t)ldq;
    float acc = 0.f;
    for (int q = lane; q < Q; q += 32) acc = fmaf(tanhf(row[q]), w2[q], acc);
    acc = warp_sum(acc);
    if (lane == 0) pa[s] = expf(acc + b2[0]);
  }
  __syncthreads();
  if (warp == 0) {
    float t = 0.f;
    for (int s = lane; s < S; s += 32) t += pa[s];
    t = warp_sum(t);
    if (lane == 0) pa[S] = t + 1e-8f;
  }
  __syncthreads();
  const float den = pa[S];
  const float* xb = x + n * S * (size_t)C;
  for (int c = threadIdx.x; c < C; c += POOLF_THREADS) {
    float acc = 0.f;
    for (int s = 0; s < S; ++s) acc = fmaf(pa[s] / den, xb[(size_t)s * C + c], acc);
    out[n * C + c] = acc;
  }
}

}  // namespace tnr

using namespace tnr;

#define DISPATCH_VPL_F32(E, CALL)                               \
  switch ((E) / 256) {                                          \
    case 1: { constexpr int VPL = 1; CALL; break; }             \
    case 2: { constexpr int VPL = 2; CALL; break; }             \
    case 3: { constexpr int VPL = 3; CALL; break; }             \
    case 4: { constexpr int VPL = 4; CALL; break; }             \
    default: set_error("hidden size %d not supported (need 256/512/768/1024)", (E)); return 1; \
  }

static int grid_for(long long items, int threads) {
  const long long want = (items + threads - 1) / threads;
  const long long cap = (long long)num_sms() * 16;
  return (int)(want < cap ? (want > 0 ? want : 1) : cap);
}

extern "C" __attribute__((visibility("default"))) int tnr_split_bf16x3(const float* x, int rows, int K, int ldx, int layout,
                                                                      int gelu, void* out_bf16, void* stream) {
  TNR_REQUIRE(rows >= 0 && K > 0 && ldx >= K, "tnr_split_bf16x3: bad shape rows=%d K=%d ldx=%d", rows, K, ldx);
  TNR_REQUIRE(layout == TNR_SPLIT_ACT || layout == TNR_SPLIT_WEIGHT, "tnr_split_bf16x3: unknown layout %d", layout);
  if (rows == 0) return 0;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  __nv_bfloat16* out = reinterpret_cast<__nv_bfloat16*>(out_bf16);
  const bool vec = K % 4 == 0 && ldx % 4 == 0 && (uintptr_t)x % 16 == 0 && (uintptr_t)out_bf16 % 8 == 0;
  const long long items = vec ? (long long)rows * (K / 4) : (long long)rows * K;
  const int grid = grid_for(items, 256);
  if (vec) {
    if (gelu) split_bf16x3_vec4_kernel<true><<<grid, 256, 0, st>>>(x, rows, K, ldx, layout, out);
    else split_bf16x3_vec4_kernel<false><<<grid, 256, 0, st>>>(x, rows, K, ldx, layout, out);
  } else {
    if (gelu) split_bf16x3_kernel<true><<<grid, 256, 0, st>>>(x, rows, K, ldx, layout, out);
    else split_bf16x3_kernel<false><<<grid, 256, 0, st>>>(x, rows, K, ldx, layout, out);
  }
  TNR_LAUNCH_CHECK();
  return 0;
}

extern "C" __attribute__((visibility("default"))) int tnr_embed_ln_fwd_f32(const int64_t* ids, int ids_ld, int n_rows, int L, int vocab,
                                                                          const float* word, const float* pos, const float* type0,
                                                                          const float* gamma, const float* beta, float eps, int E,
                                                                          float* out, void* stream) {
  TNR_REQUIRE(E % 256 == 0, "tnr_embed_ln_fwd_f32: E=%d must be a multiple of 256", E);
  TNR_REQUIRE(n_rows >= 0 && L > 0 && vocab > 0, "tnr_embed_ln_fwd_f32: bad shape");
  TNR_REQUIRE(((uintptr_t)word | (uintptr_t)pos | (uintptr_t)type0 | (uintptr_t)gamma | (uintptr_t)beta | (uintptr_t)out) % 16 == 0,
              "tnr_embed_ln_fwd_f32: 16-byte alignment required");
  if (n_rows == 0) return 0;
  const long long T = (long long)n_rows * L;
  const int grid = (int)((T + F32_ROW_WARPS - 1) / F32_ROW_WARPS);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  DISPATCH_VPL_F32(E, (embed_ln_f32_kernel<VPL><<<grid, F32_ROW_WARPS * 32, 0, st>>>(
                          ids, ids_ld, L, T, vocab, word, pos, type0, gamma, beta, eps, out)));
  TNR_LAUNCH_CHECK();
  return 0;
}

extern "C" __attribute__((visibility("default"))) int tnr_add_layernorm_f32(const float* x, const float* residual, int rows, int E,
                                                                           const float* gamma, const float* beta, float eps, float* y,
                                                                           void* stream) {
  TNR_REQUIRE(rows >= 0, "tnr_add_layernorm_f32: bad shape");
  TNR_REQUIRE(((uintptr_t)x | (uintptr_t)residual | (uintptr_t)gamma | (uintptr_t)beta | (uintptr_t)y) % 16 == 0,
              "tnr_add_layernorm_f32: 16-byte alignment required");
  if (rows == 0) return 0;
  const int grid = (int)(((long long)rows + F32_ROW_WARPS - 1) / F32_ROW_WARPS);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  DISPATCH_VPL_F32(E, (add_ln_f32_kernel<VPL><<<grid, F32_ROW_WARPS * 32, 0, st>>>(x, residual, rows, gamma, beta, eps, y)));
  TNR_LAUNCH_CHECK();
  return 0;
}

extern "C" __attribute__((visibility("default"))) int tnr_attn_relpos_fwd_f32(const float* qkv, const int64_t* mask, int mask_ld,
                                                                             const float* relbias, float* ctx, int n_news, int L,
                                                                             int A, int E, void* stream) {
  TNR_REQUIRE(L >= 1 && L <= 512, "tnr_attn_relpos_fwd_f32: L=%d out of range (1..512)", L);
  TNR_REQUIRE(A >= 1 && E == 64 * A, "tnr_attn_relpos_fwd_f32: head dim must be 64 (E=%d, A=%d)", E, A);
  TNR_REQUIRE(n_news >= 0 && n_news <= 65535, "tnr_attn_relpos_fwd_f32: n_news=%d out of range (0..65535)", n_news);
  TNR_REQUIRE(((uintptr_t)qkv | (uintptr_t)ctx) % 16 == 0, "tnr_attn_relpos_fwd_f32: 16-byte alignment required");
  if (n_news == 0) return 0;
  dim3 grid((L + ATF_Q - 1) / ATF_Q, A, n_news);
  attn_f32_kernel<<<grid, ATF_WARPS * 32, 0, reinterpret_cast<cudaStream_t>(stream)>>>(qkv, mask, mask_ld, relbias, ctx, L, E);
  TNR_LAUNCH_CHECK();
  return 0;
}

extern "C" __attribute__((visibility("default"))) int tnr_attnpool_fwd_f32(const float* x, const float* u, int ldq, int Q, const float* w2,
                                                                          const float* b2, float* out, int n, int S, int C,
                                                                          void* stream) {
  TNR_REQUIRE(S >= 1 && S <= 512, "tnr_attnpool_fwd_f32: S=%d out of range (1..512)", S);
  TNR_REQUIRE(Q >= 1 && ldq >= Q && C >= 1, "tnr_attnpool_fwd_f32: bad shape Q=%d ldq=%d C=%d", Q, ldq, C);
  if (n == 0) return 0;
  TNR_REQUIRE(n > 0 && n <= 0x7fffffff, "tnr_attnpool_fwd_f32: bad n=%d", n);
  attnpool_f32_kernel<<<n, POOLF_THREADS, (S + 1) * sizeof(float), reinterpret_cast<cudaStream_t>(stream)>>>(
      x, u, ldq, Q, w2, b2, out, S, C);
  TNR_LAUNCH_CHECK();
  return 0;
}
