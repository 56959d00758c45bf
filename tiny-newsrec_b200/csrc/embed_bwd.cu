// Backward of the embedding + LayerNorm + dropout of the news encoder (tnr_embed_ln_fwd):
//   out = dropout(LN(word[id] + pos[l] + type[0]))          (tnlrv3/modeling.py:153-178)
// Nothing beyond the ids is saved by the forward: the LayerNorm statistics are recomputed from the gathered row and
// the dropout mask is regenerated from its Philox counter.  Every sum is formed in a fixed order (no floating-point
// atomics), so a rerun is bit-identical:
//   1. rows kernel: persistent warps bound to one position l (the forward's mapping) recompute each token's input
//      gradient dx and keep per-warp sums of dx (-> dpos, dtype), dy' xhat (-> dgamma) and dy' (-> dbeta) in registers;
//      each token's four row scalars (mean, rstd, mean(g), mean(g xhat)) go to the workspace;
//   2. two small reductions fold the per-warp sums, first over the warps of a position, then over positions;
//   3. the token ids are sorted (stable, CUB radix sort: the tokens of an id stay in token order);
//   4. word kernel: a warp per chunk of EB_CHUNK sorted tokens recomputes dx from the saved scalars and sums each id's
//      run in token order.  A run that lies inside one chunk is added to dword[id] directly; the pieces of a run that
//      crosses chunk boundaries (the hot ids [CLS] / [SEP] are in every row) are parked per chunk, and
//   5. a fix-up kernel adds them up in chunk order.  Every dword row has exactly one writer.
// Pad tokens (id 0) feed dpos / dtype / dgamma / dbeta but not dword (nn.Embedding(padding_idx=0)).
#include "common.cuh"
#include <cub/device/device_radix_sort.cuh>

namespace tnr {

constexpr int EB_WARPS = 8;            // warps per block of the rows and word kernels
constexpr int EB_TARGET_WARPS = 2048;  // rows kernel: groups = 2048 / L warps per position (device-independent order)
constexpr int EB_CHUNK = 32;           // sorted tokens per warp of the word kernel

// 8 consecutive fp32 values (two 16-byte loads)
__device__ __forceinline__ void load8f(float (&v)[8], const float* p) {
  const float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + 4);
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}

// The forward's pre-LN row x = word[id] + (pos[l] + type0) and the gradient at the LayerNorm output dyd = dy * keep /
// (1 - p) of token t; lane owns columns (v * 32 + lane) * 8 + [0, 8) as in the forward.
template <int VPL, bool WORD_BF16>
__device__ __forceinline__ void eb_load_token(float (&x)[VPL * 8], float (&dyd)[VPL * 8], const void* __restrict__ word,
                                              long long id, const float* __restrict__ pos, const float* __restrict__ type0,
                                              const __nv_bfloat16* __restrict__ dy, size_t t, int l, const DropCfg& dc,
                                              int lane) {
  constexpr int E = VPL * 256;
#pragma unroll
  for (int v = 0; v < VPL; ++v) {
    const int col = (v * 32 + lane) * 8;
    float w[8], p[8], ty[8];
    if (WORD_BF16) {
      unpack8(*reinterpret_cast<const bf16x8*>(reinterpret_cast<const __nv_bfloat16*>(word) + (size_t)id * E + col), w);
    } else {
      load8f(w, reinterpret_cast<const float*>(word) + (size_t)id * E + col);
    }
    load8f(p, pos + (size_t)l * E + col);
    load8f(ty, type0 + col);
#pragma unroll
    for (int i = 0; i < 8; ++i) x[v * 8 + i] = w[i] + (p[i] + ty[i]);
    float d[8];
    unpack8(*reinterpret_cast<const bf16x8*>(dy + t * E + col), d);
    if (dc.thr16 != 0) {
      f32x2 m[4];
      dropout_mul8(dc, ((uint64_t)t * (uint64_t)E + (uint64_t)col) >> 3, m);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float m0, m1;
        upk2(m[i], m0, m1);
        d[2 * i] *= m0;
        d[2 * i + 1] *= m1;
      }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) dyd[v * 8 + i] = d[i];
  }
}

// dx = rstd * (g - mean(g) - xhat * mean(g xhat)), g = dyd * gamma, xhat = (x - mean) * rstd
template <int VPL>
__device__ __forceinline__ void eb_dx(float (&dx)[VPL * 8], const float (&x)[VPL * 8], const float (&dyd)[VPL * 8],
                                      const float* __restrict__ gamma, float mean, float rstd, float sg, float sgx, int lane) {
#pragma unroll
  for (int v = 0; v < VPL; ++v) {
    float gm[8];
    load8f(gm, gamma + (v * 32 + lane) * 8);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float xh = (x[v * 8 + i] - mean) * rstd;
      dx[v * 8 + i] = rstd * ((dyd[v * 8 + i] * gm[i] - sg) - xh * sgx);
    }
  }
}

__device__ __forceinline__ long long eb_clamp(long long id, int vocab) { return id < 0 ? 0 : (id >= vocab ? vocab - 1 : id); }

// part[w][3][E] = this warp's sums of {dx, dyd xhat, dyd} over its tokens (w = grp * L + l); stats[t] = row scalars
template <int VPL, bool WORD_BF16>
__global__ void __launch_bounds__(EB_WARPS * 32)
embed_bwd_rows_kernel(const int64_t* __restrict__ ids, int ids_ld, int L, int n_rows, int groups, int vocab,
                      const void* __restrict__ word, const float* __restrict__ pos, const float* __restrict__ type0,
                      const float* __restrict__ gamma, float eps, const __nv_bfloat16* __restrict__ dy,
                      float* __restrict__ part, float4* __restrict__ stats, const tnr_dropout drop) {
  constexpr int E = VPL * 256;
  const int warp = uniform_warp_id(), lane = threadIdx.x & 31;
  const int w = blockIdx.x * EB_WARPS + warp;
  const int l = w % L, grp = w / L;
  if (grp >= groups) return;
  const DropCfg dc = load_drop(drop);
  float adx[VPL * 8], adg[VPL * 8], adb[VPL * 8];
#pragma unroll
  for (int i = 0; i < VPL * 8; ++i) { adx[i] = 0.f; adg[i] = 0.f; adb[i] = 0.f; }
  for (int n = grp; n < n_rows; n += groups) {
    const size_t t = (size_t)n * L + l;
    const long long id = eb_clamp(ids[(size_t)n * ids_ld + l], vocab);
    float x[VPL * 8], dyd[VPL * 8];
    eb_load_token<VPL, WORD_BF16>(x, dyd, word, id, pos, type0, dy, t, l, dc, lane);
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < VPL * 8; ++i) s += x[i];
    const float mean = warp_sum(s) * (1.0f / E);
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < VPL * 8; ++i) { const float d = x[i] - mean; q = fmaf(d, d, q); }
    const float rstd = rsqrtf(warp_sum(q) * (1.0f / E) + eps);
    float sg = 0.f, sgx = 0.f;
#pragma unroll
    for (int v = 0; v < VPL; ++v) {
      float gm[8];
      load8f(gm, gamma + (v * 32 + lane) * 8);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float xh = (x[v * 8 + i] - mean) * rstd;
        const float g = dyd[v * 8 + i] * gm[i];
        sg += g;
        sgx = fmaf(g, xh, sgx);
        adg[v * 8 + i] = fmaf(dyd[v * 8 + i], xh, adg[v * 8 + i]);
        adb[v * 8 + i] += dyd[v * 8 + i];
      }
    }
    sg = warp_sum(sg) * (1.0f / E);
    sgx = warp_sum(sgx) * (1.0f / E);
    float dx[VPL * 8];
    eb_dx<VPL>(dx, x, dyd, gamma, mean, rstd, sg, sgx, lane);
#pragma unroll
    for (int i = 0; i < VPL * 8; ++i) adx[i] += dx[i];
    if (lane == 0) stats[t] = make_float4(mean, rstd, sg, sgx);
  }
  float* pw = part + (size_t)w * 3 * E;
#pragma unroll
  for (int v = 0; v < VPL; ++v) {
    const int col = (v * 32 + lane) * 8;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int i = v * 8 + 4 * h;
      *reinterpret_cast<float4*>(pw + col + 4 * h) = make_float4(adx[i], adx[i + 1], adx[i + 2], adx[i + 3]);
      *reinterpret_cast<float4*>(pw + E + col + 4 * h) = make_float4(adg[i], adg[i + 1], adg[i + 2], adg[i + 3]);
      *reinterpret_cast<float4*>(pw + 2 * E + col + 4 * h) = make_float4(adb[i], adb[i + 1], adb[i + 2], adb[i + 3]);
    }
  }
}

// red[l][c] = sum over grp (in order) of part[grp * L + l][c], c < 3E; dpos[l][c] += red[l][c] for c < E
__global__ void __launch_bounds__(256)
embed_bwd_pos_kernel(const float* __restrict__ part, int L, int groups, int E, float* __restrict__ red,
                     float* __restrict__ dpos) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int C = 3 * E;
  if (idx >= (long long)L * C) return;
  const int l = (int)(idx / C), c = (int)(idx % C);
  float s = 0.f;
  for (int grp = 0; grp < groups; ++grp) s += part[((size_t)grp * L + l) * C + c];
  red[idx] = s;
  if (dpos != nullptr && c < E) dpos[(size_t)l * E + c] += s;
}

// sum over positions (in order) of red[l][c]: c < E -> dtype0, E <= c < 2E -> dgamma, 2E <= c < 3E -> dbeta
__global__ void __launch_bounds__(256)
embed_bwd_col_kernel(const float* __restrict__ red, int L, int E, float* __restrict__ dtype0, float* __restrict__ dgamma,
                     float* __restrict__ dbeta) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= 3 * E) return;
  float* dst = c < E ? dtype0 : (c < 2 * E ? dgamma : dbeta);
  if (dst == nullptr) return;
  float s = 0.f;
  for (int l = 0; l < L; ++l) s += red[(size_t)l * 3 * E + c];
  dst[c % E] += s;
}

// sort input: clamped ids as keys, token indices as values; chunk flags reset (the fix-up reads them)
__global__ void __launch_bounds__(256)
embed_bwd_keys_kernel(const int64_t* __restrict__ ids, int ids_ld, int L, long long T, int vocab, int* __restrict__ keys,
                      int* __restrict__ vals, int* __restrict__ head_id, int* __restrict__ tail_id, int n_chunks) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < T) {
    keys[t] = (int)eb_clamp(ids[(size_t)(t / L) * ids_ld + t % L], vocab);
    vals[t] = (int)t;
  }
  if (t < n_chunks) { head_id[t] = -1; tail_id[t] = -1; }
}

template <int VPL>
__device__ __forceinline__ void eb_store_row(float* __restrict__ dst, const float (&a)[VPL * 8], bool accumulate, int lane) {
#pragma unroll
  for (int v = 0; v < VPL; ++v) {
    const int col = (v * 32 + lane) * 8;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      float4* p = reinterpret_cast<float4*>(dst + col + 4 * h);
      const int i = v * 8 + 4 * h;
      float4 o = make_float4(a[i], a[i + 1], a[i + 2], a[i + 3]);
      if (accumulate) {
        const float4 c = *p;
        o = make_float4(c.x + o.x, c.y + o.y, c.z + o.z, c.w + o.w);
      }
      *p = o;
    }
  }
}

template <int VPL, bool WORD_BF16>
__global__ void __launch_bounds__(EB_WARPS * 32)
embed_bwd_word_kernel(const int* __restrict__ keys, const int* __restrict__ vals, long long T, int L, const void* __restrict__ word,
                      const float* __restrict__ pos, const float* __restrict__ type0, const float* __restrict__ gamma,
                      const __nv_bfloat16* __restrict__ dy, const float4* __restrict__ stats, float* __restrict__ dword,
                      float* __restrict__ head, float* __restrict__ tail, int* __restrict__ head_id, int* __restrict__ tail_id,
                      int n_chunks, const tnr_dropout drop) {
  constexpr int E = VPL * 256;
  const int warp = uniform_warp_id(), lane = threadIdx.x & 31;
  const int c = blockIdx.x * EB_WARPS + warp;
  if (c >= n_chunks) return;
  const long long k0 = (long long)c * EB_CHUNK;
  const long long k1 = k0 + EB_CHUNK < T ? k0 + EB_CHUNK : T;
  if (keys[k1 - 1] == 0) return;                          // pad tokens only (they sort first)
  const DropCfg dc = load_drop(drop);
  const int before = k0 > 0 ? keys[k0 - 1] : -1;          // id of the run that may enter this chunk
  const int after = k1 < T ? keys[k1] : -1;               // id of the run that may leave it
  float acc[VPL * 8];
  int cur = -1;
  auto flush = [&]() {
    if (cur <= 0) return;
    if (cur == before) {                                  // the run began in an earlier chunk (it may go on after this one)
      eb_store_row<VPL>(head + (size_t)c * E, acc, false, lane);
      if (lane == 0) head_id[c] = cur;
    } else if (cur == after) {                            // begins here, goes on: this chunk owns the run's fix-up
      eb_store_row<VPL>(tail + (size_t)c * E, acc, false, lane);
      if (lane == 0) tail_id[c] = cur;
    } else {
      eb_store_row<VPL>(dword + (size_t)cur * E, acc, true, lane);
    }
  };
  for (long long k = k0; k < k1; ++k) {
    const int id = keys[k];
    if (id == 0) continue;
    if (id != cur) {
      flush();
      cur = id;
#pragma unroll
      for (int i = 0; i < VPL * 8; ++i) acc[i] = 0.f;
    }
    const size_t t = (size_t)vals[k];
    const int l = (int)(t % L);
    float x[VPL * 8], dyd[VPL * 8], dx[VPL * 8];
    eb_load_token<VPL, WORD_BF16>(x, dyd, word, id, pos, type0, dy, t, l, dc, lane);
    const float4 st = stats[t];
    eb_dx<VPL>(dx, x, dyd, gamma, st.x, st.y, st.z, st.w, lane);
#pragma unroll
    for (int i = 0; i < VPL * 8; ++i) acc[i] += dx[i];
  }
  flush();
}

// runs that cross chunk boundaries: the owning chunk's piece, then the pieces of the following chunks, in chunk order
template <int VPL>
__global__ void __launch_bounds__(EB_WARPS * 32)
embed_bwd_fixup_kernel(const float* __restrict__ head, const float* __restrict__ tail, const int* __restrict__ head_id,
                       const int* __restrict__ tail_id, int n_chunks, float* __restrict__ dword) {
  constexpr int E = VPL * 256;
  const int warp = uniform_warp_id(), lane = threadIdx.x & 31;
  const int c = blockIdx.x * EB_WARPS + warp;
  if (c >= n_chunks) return;
  const int id = tail_id[c];
  if (id <= 0) return;
  float acc[VPL * 8];
#pragma unroll
  for (int v = 0; v < VPL; ++v) {
    float a[8];
    load8f(a, tail + (size_t)c * E + (v * 32 + lane) * 8);
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[v * 8 + i] = a[i];
  }
  for (int cc = c + 1; cc < n_chunks && head_id[cc] == id; ++cc) {
#pragma unroll
    for (int v = 0; v < VPL; ++v) {
      float a[8];
      load8f(a, head + (size_t)cc * E + (v * 32 + lane) * 8);
#pragma unroll
      for (int i = 0; i < 8; ++i) acc[v * 8 + i] += a[i];
    }
  }
  eb_store_row<VPL>(dword + (size_t)id * E, acc, true, lane);
}

// workspace layout (every piece 256-byte aligned)
struct EbLayout {
  size_t part, red, stats, keys_in, keys_out, vals_in, vals_out, head, tail, head_id, tail_id, cub, total;
  size_t cub_bytes;
  int groups, n_chunks, end_bit;
};

static size_t eb_al(size_t x) { return (x + 255) & ~(size_t)255; }

static int eb_layout(EbLayout& lay, int n_rows, int L, int vocab, int E) {
  const long long T = (long long)n_rows * L;
  int groups = EB_TARGET_WARPS / L;
  if (groups < 1) groups = 1;
  if (groups > n_rows) groups = n_rows;
  lay.groups = groups;
  lay.n_chunks = (int)((T + EB_CHUNK - 1) / EB_CHUNK);
  int bits = 1;
  while (bits < 31 && (1ll << bits) < (long long)vocab) ++bits;
  lay.end_bit = bits;
  size_t cub_bytes = 0;
  if (cub::DeviceRadixSort::SortPairs(nullptr, cub_bytes, (const int*)nullptr, (int*)nullptr, (const int*)nullptr,
                                      (int*)nullptr, (int)T, 0, bits) != cudaSuccess)
    return 1;
  lay.cub_bytes = cub_bytes;
  size_t off = 0;
  auto take = [&](size_t bytes) { const size_t o = off; off += eb_al(bytes); return o; };
  lay.part = take((size_t)groups * L * 3 * E * 4);
  lay.red = take((size_t)L * 3 * E * 4);
  lay.stats = take((size_t)T * 16);
  lay.keys_in = take((size_t)T * 4);
  lay.keys_out = take((size_t)T * 4);
  lay.vals_in = take((size_t)T * 4);
  lay.vals_out = take((size_t)T * 4);
  lay.head = take((size_t)lay.n_chunks * E * 4);
  lay.tail = take((size_t)lay.n_chunks * E * 4);
  lay.head_id = take((size_t)lay.n_chunks * 4);
  lay.tail_id = take((size_t)lay.n_chunks * 4);
  lay.cub = take(cub_bytes);
  lay.total = off;
  return 0;
}

}  // namespace tnr

using namespace tnr;

#define EB_DISPATCH_VPL(E, CALL)                                \
  switch ((E) / 256) {                                          \
    case 1: { constexpr int VPL = 1; CALL; break; }             \
    case 2: { constexpr int VPL = 2; CALL; break; }             \
    case 3: { constexpr int VPL = 3; CALL; break; }             \
    case 4: { constexpr int VPL = 4; CALL; break; }             \
    default: set_error("hidden size %d not supported (need 256/512/768/1024)", (E)); return 1; \
  }

extern "C" __attribute__((visibility("default"))) long long tnr_embed_ln_bwd_ws_bytes(int n_rows, int L, int vocab, int E) {
  if (n_rows < 1 || L < 1 || vocab < 1 || E < 256) return 0;
  EbLayout lay;
  if (eb_layout(lay, n_rows, L, vocab, E)) return -1;
  return (long long)lay.total;
}

extern "C" __attribute__((visibility("default"))) int tnr_embed_ln_bwd(
    const int64_t* ids, int ids_ld, int n_rows, int L, int vocab, const void* word, int word_dtype, const float* pos,
    const float* type0, const float* gamma, float eps, int E, const void* dy_bf16, float* dword, float* dpos, float* dtype0,
    float* dgamma, float* dbeta, void* workspace, long long ws_bytes, const tnr_dropout* drop, void* stream) {
  TNR_REQUIRE(E % 256 == 0 && E >= 256 && E <= 1024, "tnr_embed_ln_bwd: E=%d must be 256, 512, 768 or 1024", E);
  TNR_REQUIRE(n_rows >= 0 && L > 0 && vocab > 0, "tnr_embed_ln_bwd: bad shape");
  TNR_REQUIRE((dgamma == nullptr) == (dbeta == nullptr), "tnr_embed_ln_bwd: dgamma and dbeta go together");
  TNR_REQUIRE((long long)n_rows * L < (1ll << 31), "tnr_embed_ln_bwd: too many tokens");
  if (n_rows == 0) return 0;
  EbLayout lay;
  TNR_REQUIRE(eb_layout(lay, n_rows, L, vocab, E) == 0, "tnr_embed_ln_bwd: radix sort size query failed");
  TNR_REQUIRE(workspace != nullptr && ws_bytes >= (long long)lay.total,
              "tnr_embed_ln_bwd: workspace of %lld bytes needed (tnr_embed_ln_bwd_ws_bytes), got %lld", (long long)lay.total,
              ws_bytes);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
  float* part = reinterpret_cast<float*>(ws + lay.part);
  float* red = reinterpret_cast<float*>(ws + lay.red);
  float4* stats = reinterpret_cast<float4*>(ws + lay.stats);
  const __nv_bfloat16* dy = reinterpret_cast<const __nv_bfloat16*>(dy_bf16);
  const tnr_dropout dr = drop_or_none(drop);
  const bool wbf = word_dtype == TNR_BF16;
  const bool need_rows = dpos != nullptr || dtype0 != nullptr || dgamma != nullptr || dword != nullptr;
  if (!need_rows) return 0;
  const int rows_grid = (lay.groups * L + EB_WARPS - 1) / EB_WARPS;
  if (wbf) {
    EB_DISPATCH_VPL(E, (embed_bwd_rows_kernel<VPL, true><<<rows_grid, EB_WARPS * 32, 0, st>>>(
                           ids, ids_ld, L, n_rows, lay.groups, vocab, word, pos, type0, gamma, eps, dy, part, stats, dr)));
  } else {
    EB_DISPATCH_VPL(E, (embed_bwd_rows_kernel<VPL, false><<<rows_grid, EB_WARPS * 32, 0, st>>>(
                           ids, ids_ld, L, n_rows, lay.groups, vocab, word, pos, type0, gamma, eps, dy, part, stats, dr)));
  }
  TNR_LAUNCH_CHECK();
  if (dpos != nullptr || dtype0 != nullptr || dgamma != nullptr) {
    const long long n_pos = (long long)L * 3 * E;
    embed_bwd_pos_kernel<<<(unsigned)((n_pos + 255) / 256), 256, 0, st>>>(part, L, lay.groups, E, red, dpos);
    TNR_LAUNCH_CHECK();
    if (dtype0 != nullptr || dgamma != nullptr) {
      embed_bwd_col_kernel<<<(3 * E + 255) / 256, 256, 0, st>>>(red, L, E, dtype0, dgamma, dbeta);
      TNR_LAUNCH_CHECK();
    }
  }
  if (dword == nullptr) return 0;
  const long long T = (long long)n_rows * L;
  int* keys_in = reinterpret_cast<int*>(ws + lay.keys_in);
  int* keys_out = reinterpret_cast<int*>(ws + lay.keys_out);
  int* vals_in = reinterpret_cast<int*>(ws + lay.vals_in);
  int* vals_out = reinterpret_cast<int*>(ws + lay.vals_out);
  float* head = reinterpret_cast<float*>(ws + lay.head);
  float* tail = reinterpret_cast<float*>(ws + lay.tail);
  int* head_id = reinterpret_cast<int*>(ws + lay.head_id);
  int* tail_id = reinterpret_cast<int*>(ws + lay.tail_id);
  const long long n_init = T > lay.n_chunks ? T : lay.n_chunks;
  embed_bwd_keys_kernel<<<(unsigned)((n_init + 255) / 256), 256, 0, st>>>(ids, ids_ld, L, T, vocab, keys_in, vals_in, head_id,
                                                                           tail_id, lay.n_chunks);
  TNR_LAUNCH_CHECK();
  size_t cub_bytes = lay.cub_bytes;
  TNR_CHECK_CUDA(cub::DeviceRadixSort::SortPairs(ws + lay.cub, cub_bytes, keys_in, keys_out, vals_in, vals_out, (int)T, 0,
                                                 lay.end_bit, st));
  const int word_grid = (lay.n_chunks + EB_WARPS - 1) / EB_WARPS;
  if (wbf) {
    EB_DISPATCH_VPL(E, (embed_bwd_word_kernel<VPL, true><<<word_grid, EB_WARPS * 32, 0, st>>>(
                           keys_out, vals_out, T, L, word, pos, type0, gamma, dy, stats, dword, head, tail, head_id, tail_id,
                           lay.n_chunks, dr)));
  } else {
    EB_DISPATCH_VPL(E, (embed_bwd_word_kernel<VPL, false><<<word_grid, EB_WARPS * 32, 0, st>>>(
                           keys_out, vals_out, T, L, word, pos, type0, gamma, dy, stats, dword, head, tail, head_id, tail_id,
                           lay.n_chunks, dr)));
  }
  TNR_LAUNCH_CHECK();
  EB_DISPATCH_VPL(E, (embed_bwd_fixup_kernel<VPL><<<word_grid, EB_WARPS * 32, 0, st>>>(head, tail, head_id, tail_id,
                                                                                       lay.n_chunks, dword)));
  TNR_LAUNCH_CHECK();
  return 0;
}
