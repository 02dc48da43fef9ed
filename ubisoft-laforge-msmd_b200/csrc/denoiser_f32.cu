// fp32-grade variants of the denoiser's non-GEMM kernels (precision 1 / the last steps of the hybrid
// schedule).  Same math as denoiser_kernels.cu with fp32 activations end to end; the GEMMs around them are
// the tf32x3 tcgen05 path.  Throughput is secondary here: this mode exists to meet the fp32 tolerance
// (<= 1e-5 per sampling step) and to cover the last sampling steps where bf16 rounding of x0_hat is no
// longer damped by c1(t).
#include "denoiser_kernels.cuh"
#include "profile.cuh"

namespace msmd {

namespace {
__device__ __forceinline__ float wsum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float wmax(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

template <int D>
__device__ __forceinline__ void ln_row_f32(float (&v)[D / 32], const float* __restrict__ g, const float* __restrict__ b,
                                           int lane) {
  constexpr int NV = D / 32;
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) s += v[i];
  const float mean = wsum(s) * (1.0f / D);
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) { const float dl = v[i] - mean; q = fmaf(dl, dl, q); }
  const float rstd = 1.0f / sqrtf(wsum(q) * (1.0f / D) + 1e-5f);
#pragma unroll
  for (int i = 0; i < NV / 4; ++i) {
    const float4 gg = *reinterpret_cast<const float4*>(g + i * 128 + lane * 4);
    const float4 bb = *reinterpret_cast<const float4*>(b + i * 128 + lane * 4);
    v[4 * i + 0] = (v[4 * i + 0] - mean) * rstd * gg.x + bb.x;
    v[4 * i + 1] = (v[4 * i + 1] - mean) * rstd * gg.y + bb.y;
    v[4 * i + 2] = (v[4 * i + 2] - mean) * rstd * gg.z + bb.z;
    v[4 * i + 3] = (v[4 * i + 3] - mean) * rstd * gg.w + bb.w;
  }
}
__device__ __forceinline__ void ld16(float (&v)[16], const float* p, int lane, bool add) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float4 t = *reinterpret_cast<const float4*>(p + i * 128 + lane * 4);
    if (add) { v[4 * i] += t.x; v[4 * i + 1] += t.y; v[4 * i + 2] += t.z; v[4 * i + 3] += t.w; }
    else { v[4 * i] = t.x; v[4 * i + 1] = t.y; v[4 * i + 2] = t.z; v[4 * i + 3] = t.w; }
  }
}
__device__ __forceinline__ void st16(float* p, const float (&v)[16], int lane) {
#pragma unroll
  for (int i = 0; i < 4; ++i)
    *reinterpret_cast<float4*>(p + i * 128 + lane * 4) = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
}
}  // namespace

// ---------------------------------------------------------------------------------------- embeddings (fp32 out)
__global__ void embed_f32_kernel(EmbedParams p, float* __restrict__ out) {
  // one block per (sequence, token); feature_proj recomputed per sequence (precision path: simplicity over speed)
  const int T = 1 + p.Lp + p.L;
  const int s = blockIdx.x / T, i = blockIdx.x % T;
  const int t = p.steps[s];
  __shared__ float xin[80];
  const int n = s % p.NX;
  if (i > p.Lp) {
    const int l = i - 1 - p.Lp;
    for (int k = threadIdx.x; k <= p.dm; k += blockDim.x)
      xin[k] = k < p.dm ? p.x[((int64_t)n * p.L + l) * p.dm + k] : (p.indicator ? p.indicator[(int64_t)s * p.L + l] : 0.f);
  }
  __syncthreads();
  for (int c = threadIdx.x; c < p.d; c += blockDim.x) {
    float v = p.PE[i * p.d + c];
    if (i == 0) v += p.pp[(int64_t)s * p.d + c] + p.temb[(int64_t)t * p.d + c];
    else if (i <= p.Lp) v += p.pmproj[((int64_t)s * p.Lp + (i - 1)) * p.d + c];
    else {
      float acc = p.bf[c];
      for (int k = 0; k <= p.dm; ++k) acc = fmaf(xin[k], p.WfT[(int64_t)k * p.d + c], acc);
      v += acc;
    }
    out[((int64_t)s * T + i) * p.d + c] = v;
  }
}
int embed_f32_launch(const EmbedParams& p, float* out, cudaStream_t st) {
  ProfileScope prof("embed_f32", st);
  embed_f32_kernel<<<p.S * (1 + p.Lp + p.L), 128, 0, st>>>(p, out);
  MSMD_CHECK_LAUNCH();
  return MSMD_OK;
}

// ---------------------------------------------------------------------------------------- LayerNorm chain (fp32)
__global__ void __launch_bounds__(256) ln_f32_kernel(const float* __restrict__ y, const float* resid,
                                                     const float* __restrict__ g1, const float* __restrict__ b1,
                                                     const float* __restrict__ add, const float* __restrict__ g2,
                                                     const float* __restrict__ b2, float* out, float* __restrict__ x0,
                                                     int M, int T) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= M) return;
  const int s = row / T, tok = row % T;
  float v[16];
  ld16(v, y + (int64_t)row * 512, lane, false);
  if (resid) ld16(v, resid + (int64_t)row * 512, lane, true);
  ln_row_f32<512>(v, g1, b1, lane);
  if (tok == 0 && x0 != nullptr) { st16(x0 + (int64_t)s * 512, v, lane); return; }
  if (add != nullptr && tok > 0) {
    ld16(v, add + ((int64_t)s * (T - 1) + (tok - 1)) * 512, lane, true);
    ln_row_f32<512>(v, g2, b2, lane);
  }
  st16(out + (int64_t)row * 512, v, lane);
}
int ln_f32_launch(const float* y, const float* resid, const float* g1, const float* b1, const float* add, const float* g2,
                  const float* b2, float* out, float* x0, int M, int T, cudaStream_t st) {
  ProfileScope prof("ln_f32", st);
  ln_f32_kernel<<<cdiv(M, 8), 256, 0, st>>>(y, resid, g1, b1, add, g2, b2, out, x0, M, T);
  MSMD_CHECK_LAUNCH();
  return MSMD_OK;
}
__global__ void __launch_bounds__(256) ln_row0_f32_kernel(const float* __restrict__ y0, const float* __restrict__ r0,
                                                          const float* __restrict__ g, const float* __restrict__ b,
                                                          float* __restrict__ out, int S, int T) {
  const int lane = threadIdx.x & 31;
  const int s = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (s >= S) return;
  float v[16];
  ld16(v, y0 + (int64_t)s * 512, lane, false);
  ld16(v, r0 + (int64_t)s * 512, lane, true);
  ln_row_f32<512>(v, g, b, lane);
  st16(out + (int64_t)s * T * 512, v, lane);
}
int ln_row0_f32_launch(const float* y0, const float* r0, const float* g, const float* b, float* out, int S, int T,
                       cudaStream_t st) {
  ln_row0_f32_kernel<<<cdiv(S, 8), 256, 0, st>>>(y0, r0, g, b, out, S, T);
  MSMD_CHECK_LAUNCH();
  return MSMD_OK;
}

// ---------------------------------------------------------------------------------------- attention (fp32, SIMT)
// one CTA per (sequence, head); thread = query row; K and V rows broadcast from shared memory; online softmax.
// q rows s*T.. (row stride ldq), k|v rows s*Tk.. (row stride ldkv, K at column h*64, V at d + h*64).  width 0: every key
// visible (self-attention); width >= 1: the alignment band of the cross attention (token 0 sees every key, token i >= 1
// the keys j with |j - (i-1)| <= width-1).
__global__ void __launch_bounds__(128) attn_f32_kernel(const float* __restrict__ q_src, int ldq, const float* __restrict__ kv,
                                                       int ldkv, float* __restrict__ ctx, int T, int Tk, int H, int width) {
  extern __shared__ float sm[];  // K [Tk][64], V [Tk][64]
  const int h = blockIdx.x, s = blockIdx.y, d = H * 64;
  float* sK = sm;
  float* sV = sm + Tk * 64;
  const float* kbase = kv + (int64_t)s * Tk * ldkv + h * 64;
  for (int i = threadIdx.x; i < Tk * 16; i += blockDim.x) {
    const int r = i >> 4, c4 = i & 15;
    *reinterpret_cast<float4*>(sK + r * 64 + c4 * 4) = *reinterpret_cast<const float4*>(kbase + (int64_t)r * ldkv + c4 * 4);
    *reinterpret_cast<float4*>(sV + r * 64 + c4 * 4) = *reinterpret_cast<const float4*>(kbase + (int64_t)r * ldkv + d + c4 * 4);
  }
  __syncthreads();
  const int i = threadIdx.x;
  if (i >= T) return;
  int j0 = 0, j1 = Tk - 1;
  if (width > 0 && i > 0) { j0 = max(0, i - width); j1 = min(Tk - 1, i + width - 2); }
  const float* qrow = q_src + ((int64_t)s * T + i) * ldq + h * 64;
  float q[64], o[64];
#pragma unroll
  for (int c4 = 0; c4 < 16; ++c4) {
    const float4 t = *reinterpret_cast<const float4*>(qrow + c4 * 4);
    q[4 * c4] = t.x * 0.125f; q[4 * c4 + 1] = t.y * 0.125f; q[4 * c4 + 2] = t.z * 0.125f; q[4 * c4 + 3] = t.w * 0.125f;
  }
#pragma unroll
  for (int c = 0; c < 64; ++c) o[c] = 0.f;
  float m = -INFINITY, l = 0.f;
  for (int j = j0; j <= j1; ++j) {
    float sc = 0.f;
#pragma unroll
    for (int c = 0; c < 64; ++c) sc = fmaf(q[c], sK[j * 64 + c], sc);
    if (sc > m) {   // new running maximum (rare after the first keys): rescale what has been accumulated
      const float a = expf(m - sc);
      l *= a;
#pragma unroll
      for (int c = 0; c < 64; ++c) o[c] *= a;
      m = sc;
    }
    const float pj = expf(sc - m);
    l += pj;
#pragma unroll
    for (int c = 0; c < 64; ++c) o[c] = fmaf(pj, sV[j * 64 + c], o[c]);
  }
  const float inv = 1.0f / l;
  float* dst = ctx + ((int64_t)s * T + i) * d + h * 64;
#pragma unroll
  for (int c4 = 0; c4 < 16; ++c4)
    *reinterpret_cast<float4*>(dst + c4 * 4) = make_float4(o[4 * c4] * inv, o[4 * c4 + 1] * inv, o[4 * c4 + 2] * inv, o[4 * c4 + 3] * inv);
}
namespace {
int attn_f32_launch(const float* q, int ldq, const float* kv, int ldkv, float* ctx, int S, int T, int Tk, int H, int width,
                    const char* name, cudaStream_t st) {
  static bool attr = false;
  if (!attr) {
    MSMD_CHECK_CUDA(cudaFuncSetAttribute(attn_f32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * 128 * 64 * 4));
    attr = true;
  }
  MSMD_REQUIRE(T <= 128 && Tk <= 128, "%s: %d queries / %d keys > 128", name, T, Tk);
  ProfileScope prof(name, st);
  attn_f32_kernel<<<dim3(H, S), 128, 2 * Tk * 64 * (int)sizeof(float), st>>>(q, ldq, kv, ldkv, ctx, T, Tk, H, width);
  MSMD_CHECK_LAUNCH();
  return MSMD_OK;
}
}  // namespace
int self_attn_f32_launch(const float* qkv, float* ctx, int S, int T, int H, cudaStream_t st) {
  const int d = H * 64;
  return attn_f32_launch(qkv, 3 * d, qkv + d, 3 * d, ctx, S, T, T, H, 0, "self_attn_f32", st);
}
int cross_attn_f32_launch(const float* q, const float* kv, float* ctx, int S, int T, int Tk, int H, int width,
                          cudaStream_t st) {
  MSMD_REQUIRE(T >= 2 && Tk >= T - 1 && width >= 0, "cross_attn_f32: %d queries / %d keys / width %d", T, Tk, width);
  const int d = H * 64;
  return attn_f32_launch(q, d, kv, 2 * d, ctx, S, T, Tk, H, width, "cross_attn_f32", st);
}

// person-token cross attention, fp32: one warp per (sequence, head); lane = output dims 2*lane, 2*lane+1
__global__ void __launch_bounds__(256) cross_attn_row0_f32_kernel(const float* __restrict__ q0, const float* __restrict__ kv,
                                                                  float* __restrict__ ctx0, int S, int Tk, int H) {
  const int lane = threadIdx.x & 31;
  const int w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (w >= S * H) return;
  const int s = w / H, h = w % H, d = H * 64;
  const float2 q = *reinterpret_cast<const float2*>(q0 + (int64_t)s * d + h * 64 + 2 * lane);
  float sc[4];
#pragma unroll
  for (int grp = 0; grp < 4; ++grp) {
    float mine = -INFINITY;
    for (int j0 = 0; j0 < 32; ++j0) {
      const int j = grp * 32 + j0;
      if (j >= Tk) break;
      const float2 k = *reinterpret_cast<const float2*>(kv + ((int64_t)s * Tk + j) * 2 * d + h * 64 + 2 * lane);
      const float p = wsum(q.x * k.x + q.y * k.y);
      if (j0 == lane) mine = p * 0.125f;
    }
    sc[grp] = mine;
  }
  const float m = wmax(fmaxf(fmaxf(sc[0], sc[1]), fmaxf(sc[2], sc[3])));
  float l = 0.f;
#pragma unroll
  for (int i = 0; i < 4; ++i) { sc[i] = (sc[i] == -INFINITY) ? 0.f : expf(sc[i] - m); l += sc[i]; }
  l = wsum(l);
  float oa = 0.f, ob = 0.f;
#pragma unroll
  for (int grp = 0; grp < 4; ++grp)
    for (int j0 = 0; j0 < 32; ++j0) {
      const int j = grp * 32 + j0;
      if (j >= Tk) break;
      const float p = __shfl_sync(0xffffffffu, sc[grp], j0);
      const float2 v = *reinterpret_cast<const float2*>(kv + ((int64_t)s * Tk + j) * 2 * d + d + h * 64 + 2 * lane);
      oa = fmaf(p, v.x, oa);
      ob = fmaf(p, v.y, ob);
    }
  *reinterpret_cast<float2*>(ctx0 + (int64_t)s * d + h * 64 + 2 * lane) = make_float2(oa / l, ob / l);
}
int cross_attn_row0_f32_launch(const float* q0, const float* kv, float* ctx0, int S, int Tk, int H, cudaStream_t st) {
  MSMD_REQUIRE(Tk <= 128, "cross_attn_row0_f32: memory length %d > 128", Tk);
  ProfileScope prof("cross_attn_row0_f32", st);
  cross_attn_row0_f32_kernel<<<cdiv(S * H, 8), 256, 0, st>>>(q0, kv, ctx0, S, Tk, H);
  MSMD_CHECK_LAUNCH();
  return MSMD_OK;
}

// memory = cat(prev_audio, audio) in fp32
__global__ void build_memory_f32_kernel(const float* __restrict__ prev_audio, const float* __restrict__ audio,
                                        float* __restrict__ mem, int S, int Lp, int L, int d) {
  const int64_t n = (int64_t)S * (Lp + L) * d;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % d);
    const int64_t row = i / d;
    const int tok = (int)(row % (Lp + L));
    const int64_t s = row / (Lp + L);
    mem[i] = tok < Lp ? prev_audio[(s * Lp + tok) * d + c] : audio[(s * L + tok - Lp) * d + c];
  }
}
int build_memory_f32(const float* prev_audio, const float* audio, float* mem, int S, int Lp, int L, int d, cudaStream_t st) {
  const int64_t n = (int64_t)S * (Lp + L) * d;
  build_memory_f32_kernel<<<(int)std::min<int64_t>(cdiv(n, 256), kNumSMs * 16), 256, 0, st>>>(prev_audio, audio, mem, S, Lp, L, d);
  MSMD_CHECK_LAUNCH();
  return MSMD_OK;
}

}  // namespace msmd
