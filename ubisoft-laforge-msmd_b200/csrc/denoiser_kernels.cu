// Non-GEMM kernels of the denoiser / sampler: embeddings (model.py:931-949), LayerNorm chains of the
// post-LN decoder layers, self-attention over the 111-token sequence, the person-token (row 0) cross
// attention, and the fused CFG-combine + static-basis mix + DDPM posterior step (model.py:404-430,
// :964-995).  All HBM-bound elementwise / small-tile work: coalesced float4 / bf16x4 accesses,
// warp-shuffle reductions, fp32 statistics.
#include "denoiser_kernels.cuh"
#include "profile.cuh"
#include <cuda_fp16.h>
#include <cstdlib>

namespace msmd {

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&h);
}
// 16-bit activation storage comes in two formats: bf16 (F16 = false) and fp16 (F16 = true, the sampler's
// intermediate-precision steps).  Buffers are typed bf16* either way; these helpers do the (un)packing.
template <bool F16>
__device__ __forceinline__ uint32_t pack_h(float lo, float hi) {
  if constexpr (F16) {
    __half2 h = __floats2half2_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&h);
  } else {
    return pack_bf16(lo, hi);
  }
}
template <bool F16>
__device__ __forceinline__ float2 unpack_h(uint32_t w) {
  if constexpr (F16) return __half22float2(*reinterpret_cast<const __half2*>(&w));
  else return make_float2(__uint_as_float(w << 16), __uint_as_float(w & 0xffff0000u));
}
template <bool F16>
__device__ __forceinline__ void store_h1(bf16* dst, float v) {
  if constexpr (F16) *reinterpret_cast<__half*>(dst) = __float2half_rn(v);
  else *dst = __float2bfloat16_rn(v);
}
__device__ __forceinline__ float gelu_exact(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752f)); }

// ------------------------------------------------------------------------------------------- small fp32 linear
__global__ void __launch_bounds__(256) linear_simt_kernel(const float* __restrict__ x, int64_t ldx,
                                                          const float* __restrict__ W, int64_t ldw,
                                                          const float* __restrict__ b, float* __restrict__ out,
                                                          int64_t ldo, int R, int C, int K, int act) {
  const int lane = threadIdx.x & 31;
  const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (w >= (int64_t)R * C) return;
  const int r = (int)(w / C), c = (int)(w % C);
  const float* xr = x + r * ldx;
  const float* wr = W + (int64_t)c * ldw;
  float s = 0.f;
  for (int k = lane; k < K; k += 32) s = fmaf(xr[k], wr[k], s);
  s = warp_sum(s);
  if (lane == 0) {
    s += b ? b[c] : 0.f;
    if (act == 1) s = gelu_exact(s);
    out[r * ldo + c] = s;
  }
}
int linear_simt(const float* x, int64_t ldx, const float* W, int64_t ldw, const float* b, float* out, int64_t ldo, int R,
                int C, int K, int act, cudaStream_t st) {
  if (R <= 0 || C <= 0) return MSMD_OK;
  const int64_t warps = (int64_t)R * C;
  linear_simt_kernel<<<cdiv(warps * 32, 256), 256, 0, st>>>(x, ldx, W, ldw, b, out, ldo, R, C, K, act);
  MSMD_CHECK_LAUNCH();
  return MSMD_OK;
}

__global__ void cast_rows_bf16_kernel(const float* __restrict__ src, int64_t lds, bf16* __restrict__ dst, int64_t ldd,
                                      int64_t rows, int cols) {
  const int64_t n = rows * cols;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / cols;
    const int c = (int)(i % cols);
    dst[r * ldd + c] = __float2bfloat16_rn(src[r * lds + c]);
  }
}
int cast_rows_bf16(const float* src, int64_t lds, bf16* dst, int64_t ldd, int64_t rows, int cols, cudaStream_t st) {
  if (rows * cols == 0) return MSMD_OK;
  cast_rows_bf16_kernel<<<(int)std::min<int64_t>(cdiv(rows * cols, 256), kNumSMs * 16), 256, 0, st>>>(src, lds, dst, ldd,
                                                                                                   rows, cols);
  MSMD_CHECK_LAUNCH();
  return MSMD_OK;
}

template <bool F16>
__global__ void build_memory_kernel(const float* __restrict__ prev_audio, const float* __restrict__ audio,
                                    bf16* __restrict__ mem, int S, int Lp, int L, int d) {
  const int64_t n = (int64_t)S * (Lp + L) * d;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % d);
    const int64_t row = i / d;
    const int tok = (int)(row % (Lp + L));
    const int64_t s = row / (Lp + L);
    const float v = tok < Lp ? prev_audio[(s * Lp + tok) * d + c] : audio[(s * L + tok - Lp) * d + c];
    store_h1<F16>(mem + i, v);
  }
}
int build_memory_h16(const float* prev_audio, const float* audio, bf16* mem, int S, int Lp, int L, int d, int fp16,
                     cudaStream_t st) {
  const int64_t n = (int64_t)S * (Lp + L) * d;
  const int grid = (int)std::min<int64_t>(cdiv(n, 256), kNumSMs * 16);
  if (fp16) build_memory_kernel<true><<<grid, 256, 0, st>>>(prev_audio, audio, mem, S, Lp, L, d);
  else build_memory_kernel<false><<<grid, 256, 0, st>>>(prev_audio, audio, mem, S, Lp, L, d);
  MSMD_CHECK_LAUNCH();
  return MSMD_OK;
}

// ------------------------------------------------------------------------------------------- embeddings
// rows 0..Lp: person token (+ timestep embedding) and the projected previous-motion context (one block per row; the
// blocks past the x-row blocks of the fused embed kernel below)
template <bool F16>
__device__ __forceinline__ void embed_ctx_rows(const EmbedParams& p, int row) {
  const int T = 1 + p.Lp + p.L;
  const int s = row / (p.Lp + 1), i = row % (p.Lp + 1);
  const int t = p.steps[s];
  for (int c = threadIdx.x; c < p.d; c += blockDim.x) {
    float v = p.PE[i * p.d + c];
    v += (i == 0) ? (p.pp[(int64_t)s * p.d + c] + p.temb[(int64_t)t * p.d + c])
                  : p.pmproj[((int64_t)s * p.Lp + (i - 1)) * p.d + c];
    store_h1<F16>(p.out + ((int64_t)s * T + i) * p.d + c, v);
  }
}
// rows Lp+1..: feature_proj([x_t, indicator]) + PE, computed once per x row and written to its E sequences.
// CTA = 25 frames x 512 features; the x rows sit in shared memory k-major ([k][28]) so one 128-bit broadcast
// load feeds 4 frames' FMAs (the scalar-load version was LDS-bound at 65 us; this one is FMA-issue-bound).
constexpr int kEmbedRows = 25, kEmbedPitch = 28;
template <bool F16>
__global__ void __launch_bounds__(256, 2) embed_x_kernel(EmbedParams p) {
  griddep_launch();
  griddep_wait();
  extern __shared__ __align__(16) float xs[];  // [dm][kEmbedPitch] x values (frame-minor), then [E][kEmbedPitch] indicators
  const int T = 1 + p.Lp + p.L;
  const int blocks_per_x = (p.L + kEmbedRows - 1) / kEmbedRows;
  if ((int)blockIdx.x >= p.NX * blocks_per_x) {      // context rows ride in the same launch (one launch fewer per step)
    embed_ctx_rows<F16>(p, (int)blockIdx.x - p.NX * blocks_per_x);
    return;
  }
  const int n = blockIdx.x / blocks_per_x;
  const int l0 = (blockIdx.x % blocks_per_x) * kEmbedRows;
  const int nr = min(kEmbedRows, p.L - l0);
  float* inds = xs + p.dm * kEmbedPitch;
  for (int i = threadIdx.x; i < kEmbedPitch * p.dm; i += blockDim.x) {
    const int r = i / p.dm, k = i % p.dm;      // coalesced global read, transposed shared write
    xs[k * kEmbedPitch + r] = r < nr ? p.x[((int64_t)n * p.L + l0 + r) * p.dm + k] : 0.f;
  }
  for (int i = threadIdx.x; i < p.E * kEmbedPitch; i += blockDim.x) {
    const int e = i / kEmbedPitch, r = i % kEmbedPitch;
    inds[i] = (p.indicator && r < nr) ? p.indicator[(int64_t)(e * p.NX + n) * p.L + l0 + r] : 0.f;
  }
  __syncthreads();
  for (int c = 2 * threadIdx.x; c < p.d; c += 2 * blockDim.x) {
    // accumulators start from bias + positional encoding: those 25 independent loads overlap the staging above
    // instead of sitting, one latency each, between the stores of the epilogue
    float a0[kEmbedPitch], a1[kEmbedPitch];
    const float2 bc = *reinterpret_cast<const float2*>(p.bf + c);
#pragma unroll
    for (int r = 0; r < kEmbedPitch; ++r) {
      float2 pe = make_float2(0.f, 0.f);
      if (r < nr) pe = __ldg(reinterpret_cast<const float2*>(p.PE + (int64_t)(1 + p.Lp + l0 + r) * p.d + c));
      a0[r] = bc.x + pe.x;
      a1[r] = bc.y + pe.y;
    }
    // weights for 4 k at a time: the 4 loads are issued together, so their (L1/L2) latency is paid once per 224 FMAs
    const float* wcol = p.WfT + c;
    for (int k0 = 0; k0 < p.dm; k0 += 4) {
      float2 w[4];
#pragma unroll
      for (int u = 0; u < 4; ++u)
        w[u] = k0 + u < p.dm ? __ldg(reinterpret_cast<const float2*>(wcol + (int64_t)(k0 + u) * p.d)) : make_float2(0.f, 0.f);
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        if (k0 + u < p.dm) {
          const float4* xr = reinterpret_cast<const float4*>(xs + (k0 + u) * kEmbedPitch);
#pragma unroll
          for (int q = 0; q < kEmbedPitch / 4; ++q) {
            const float4 xv = xr[q];
            a0[4 * q + 0] = fmaf(xv.x, w[u].x, a0[4 * q + 0]); a1[4 * q + 0] = fmaf(xv.x, w[u].y, a1[4 * q + 0]);
            a0[4 * q + 1] = fmaf(xv.y, w[u].x, a0[4 * q + 1]); a1[4 * q + 1] = fmaf(xv.y, w[u].y, a1[4 * q + 1]);
            a0[4 * q + 2] = fmaf(xv.z, w[u].x, a0[4 * q + 2]); a1[4 * q + 2] = fmaf(xv.z, w[u].y, a1[4 * q + 2]);
            a0[4 * q + 3] = fmaf(xv.w, w[u].x, a0[4 * q + 3]); a1[4 * q + 3] = fmaf(xv.w, w[u].y, a1[4 * q + 3]);
          }
        }
      }
    }
    const float2 wi = *reinterpret_cast<const float2*>(p.WfT + (int64_t)p.dm * p.d + c);
#pragma unroll
    for (int r = 0; r < kEmbedRows; ++r) {
      if (r < nr) {
        const int l = l0 + r;
        for (int e = 0; e < p.E; ++e) {
          const float ind = inds[e * kEmbedPitch + r];
          const int s = e * p.NX + n;
          *reinterpret_cast<uint32_t*>(p.out + ((int64_t)s * T + 1 + p.Lp + l) * p.d + c) =
              pack_h<F16>(fmaf(ind, wi.x, a0[r]), fmaf(ind, wi.y, a1[r]));
        }
      }
    }
  }
}

// The same rows on the tensor cores.  feature_proj is a [rows, dm] x [dm, 512] product with fp32 inputs (x_t is the
// sampler state) and a 16-bit output: three mma.sync passes over fp16 two-term splits (x = hi + lo, W = hi + lo:
// hi*hi + lo*hi + hi*lo, 22 mantissa bits - the result rounds to the same 16-bit value as the fp32 FMA chain except
// for rare last-bit ties) cost 240 MMAs per warp instead of 3800 FFMAs + 480 shared-memory loads per thread.
//   CTA   = 32 consecutive x rows (clip boundaries may fall inside a tile) x 512 features, 8 warps x 64 features
//   A     = the rows' hi / lo halves in shared memory (pitch 88: ldmatrix conflict-free), K zero-padded to 80
//   B     = Wf16 [n][k] fragments straight from global memory (164 KB in all: L1 / L2 resident)
//   out   = accumulators -> a warp-private fp32 staging tile -> + bias + PE (+ indicator * w_ind per guidance entry)
//           -> 16-byte stores of 8 features, one row segment of 128 bytes per 8 lanes, to each of the E sequences
constexpr int kEmRows = 32, kEmK = 80, kEmAPitch = 88, kEmSPitch = 72;
constexpr int kEmSmem = 2 * kEmRows * kEmAPitch * 2 + 3 * kEmRows * 4 + 8 * kEmRows * kEmSPitch * 4;
__device__ __forceinline__ void em_ldmatrix_x4(uint32_t (&r)[4], const void* smem_row) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"((uint32_t)__cvta_generic_to_shared(smem_row)));
}
__device__ __forceinline__ void em_mma(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3]) : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
template <bool F16>
__global__ void __launch_bounds__(256, 2) embed_x_mma_kernel(EmbedParams p) {
  griddep_launch();
  griddep_wait();
  extern __shared__ __align__(16) uint8_t esm[];
  const int T = 1 + p.Lp + p.L;
  const int rows_total = p.NX * p.L;
  const int n_tiles = (rows_total + kEmRows - 1) / kEmRows;
  if ((int)blockIdx.x >= n_tiles) {                  // context rows ride in the same launch
    embed_ctx_rows<F16>(p, (int)blockIdx.x - n_tiles);
    return;
  }
  __half* a_hi = reinterpret_cast<__half*>(esm);
  __half* a_lo = a_hi + kEmRows * kEmAPitch;
  float* inds = reinterpret_cast<float*>(a_lo + kEmRows * kEmAPitch);      // [3][32]
  float* stage = inds + 3 * kEmRows;                                         // [8 warps][32][72]
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, gid = lane >> 2, tig = lane & 3;
  const int g0 = blockIdx.x * kEmRows;
  for (int i = tid; i < kEmRows * kEmK; i += 256) {
    const int r = i / kEmK, k = i - r * kEmK;
    float v = 0.f;
    if (k < p.dm && g0 + r < rows_total) v = p.x[(int64_t)(g0 + r) * p.dm + k];
    const __half hi = __float2half_rn(v);
    a_hi[r * kEmAPitch + k] = hi;
    a_lo[r * kEmAPitch + k] = __float2half_rn(v - __half2float(hi));
  }
  for (int i = tid; i < 3 * kEmRows; i += 256) {
    const int e = i / kEmRows, r = i - e * kEmRows, g = g0 + r;
    float v = 0.f;
    if (p.indicator != nullptr && e < p.E && g < rows_total) {
      const int n = g / p.L, l = g - n * p.L;
      v = p.indicator[(int64_t)(e * p.NX + n) * p.L + l];
    }
    inds[i] = v;
  }
  __syncthreads();

  const int n0 = warp * 64;
  float acc[2][8][4];
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < 8; ++nt)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[mt][nt][j] = 0.f;
  const __half* Wh = static_cast<const __half*>(p.Wf16);
  const __half* Wl = Wh + (int64_t)p.d * kEmK;
  const int a_off = ((lane & 7) + ((lane >> 3) & 1) * 8) * kEmAPitch + (lane >> 4) * 8;
#pragma unroll
  for (int ks = 0; ks < kEmK / 16; ++ks) {
    uint32_t ah[2][4], al[2][4];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) {
      em_ldmatrix_x4(ah[mt], a_hi + 16 * mt * kEmAPitch + a_off + 16 * ks);
      em_ldmatrix_x4(al[mt], a_lo + 16 * mt * kEmAPitch + a_off + 16 * ks);
    }
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      const int64_t wo = (int64_t)(n0 + 8 * nt + gid) * kEmK + 16 * ks + 2 * tig;
      const uint32_t bh0 = __ldg(reinterpret_cast<const uint32_t*>(Wh + wo)), bh1 = __ldg(reinterpret_cast<const uint32_t*>(Wh + wo + 8));
      const uint32_t bl0 = __ldg(reinterpret_cast<const uint32_t*>(Wl + wo)), bl1 = __ldg(reinterpret_cast<const uint32_t*>(Wl + wo + 8));
#pragma unroll
      for (int mt = 0; mt < 2; ++mt) {
        em_mma(acc[mt][nt], al[mt], bh0, bh1);   // lo * hi
        em_mma(acc[mt][nt], ah[mt], bl0, bl1);   // hi * lo
        em_mma(acc[mt][nt], ah[mt], bh0, bh1);   // hi * hi
      }
    }
  }
  float* sw = stage + warp * (kEmRows * kEmSPitch);
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      *reinterpret_cast<float2*>(sw + (16 * mt + gid) * kEmSPitch + 8 * nt + 2 * tig) = make_float2(acc[mt][nt][0], acc[mt][nt][1]);
      *reinterpret_cast<float2*>(sw + (16 * mt + gid + 8) * kEmSPitch + 8 * nt + 2 * tig) = make_float2(acc[mt][nt][2], acc[mt][nt][3]);
    }
  __syncwarp();
  // lane = (row within a group of 4, 8-feature segment): 8 lanes write one 128-byte row segment per entry
  const int c8 = (lane & 7) * 8, col = n0 + c8;
  float bias[8], wi[8];
  {
    const float4 b0 = __ldg(reinterpret_cast<const float4*>(p.bf + col)), b1 = __ldg(reinterpret_cast<const float4*>(p.bf + col + 4));
    const float4 w0 = __ldg(reinterpret_cast<const float4*>(p.WfT + (int64_t)p.dm * p.d + col));
    const float4 w1 = __ldg(reinterpret_cast<const float4*>(p.WfT + (int64_t)p.dm * p.d + col + 4));
    bias[0] = b0.x; bias[1] = b0.y; bias[2] = b0.z; bias[3] = b0.w; bias[4] = b1.x; bias[5] = b1.y; bias[6] = b1.z; bias[7] = b1.w;
    wi[0] = w0.x; wi[1] = w0.y; wi[2] = w0.z; wi[3] = w0.w; wi[4] = w1.x; wi[5] = w1.y; wi[6] = w1.z; wi[7] = w1.w;
  }
  // the positional-encoding rows of all 8 row groups are requested before the first is used (the accumulators are dead
  // by now, so the registers are free): one L2 latency instead of eight on the critical path of a 200-CTA kernel
  float4 pe0[kEmRows / 4], pe1[kEmRows / 4];
#pragma unroll
  for (int it = 0; it < kEmRows / 4; ++it) {
    const int g = g0 + it * 4 + (lane >> 3);
    pe0[it] = pe1[it] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (g < rows_total) {
      const int l = g - (g / p.L) * p.L;
      const float* pe = p.PE + (int64_t)(1 + p.Lp + l) * p.d + col;
      pe0[it] = __ldg(reinterpret_cast<const float4*>(pe));
      pe1[it] = __ldg(reinterpret_cast<const float4*>(pe + 4));
    }
  }
#pragma unroll
  for (int it = 0; it < kEmRows / 4; ++it) {
    const int r = it * 4 + (lane >> 3), g = g0 + r;
    if (g < rows_total) {
      const int n = g / p.L, l = g - n * p.L;
      const float4 s0 = *reinterpret_cast<const float4*>(sw + r * kEmSPitch + c8), s1 = *reinterpret_cast<const float4*>(sw + r * kEmSPitch + c8 + 4);
      const float4 p0 = pe0[it], p1 = pe1[it];
      float v[8] = {s0.x + (bias[0] + p0.x), s0.y + (bias[1] + p0.y), s0.z + (bias[2] + p0.z), s0.w + (bias[3] + p0.w),
                    s1.x + (bias[4] + p1.x), s1.y + (bias[5] + p1.y), s1.z + (bias[6] + p1.z), s1.w + (bias[7] + p1.w)};
      for (int e = 0; e < p.E; ++e) {
        const float ind = inds[e * kEmRows + r];
        uint4 o;
        o.x = pack_h<F16>(fmaf(ind, wi[0], v[0]), fmaf(ind, wi[1], v[1]));
        o.y = pack_h<F16>(fmaf(ind, wi[2], v[2]), fmaf(ind, wi[3], v[3]));
        o.z = pack_h<F16>(fmaf(ind, wi[4], v[4]), fmaf(ind, wi[5], v[5]));
        o.w = pack_h<F16>(fmaf(ind, wi[6], v[6]), fmaf(ind, wi[7], v[7]));
        *reinterpret_cast<uint4*>(p.out + ((int64_t)(e * p.NX + n) * T + 1 + p.Lp + l) * p.d + col) = o;
      }
    }
  }
}
int embed_launch(const EmbedParams& p, cudaStream_t st) {
  ProfileScope prof("embed", st);
  static const bool use_mma = [] { const char* e = getenv("MSMD_EMBED_MMA"); return e ? atoi(e) != 0 : true; }();
  if (use_mma && p.Wf16 != nullptr && p.d == 512 && p.dm <= kEmK && p.E <= 3) {
    static bool attr = false;
    if (!attr) {
      MSMD_CHECK_CUDA(cudaFuncSetAttribute(embed_x_mma_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kEmSmem));
      MSMD_CHECK_CUDA(cudaFuncSetAttribute(embed_x_mma_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kEmSmem));
      attr = true;
    }
    const int blocks = cdiv(p.NX * p.L, kEmRows) + p.S * (p.Lp + 1);
    MSMD_CHECK_CUDA(launch_pdl(p.fp16 ? embed_x_mma_kernel<true> : embed_x_mma_kernel<false>, dim3(blocks), dim3(256), kEmSmem, st, p));
    MSMD_CHECK_LAUNCH();
    return MSMD_OK;
  }
  const int blocks = p.NX * ((p.L + kEmbedRows - 1) / kEmbedRows) + p.S * (p.Lp + 1);
  MSMD_CHECK_CUDA(launch_pdl(p.fp16 ? embed_x_kernel<true> : embed_x_kernel<false>, dim3(blocks), dim3(256),
                             (p.dm + 3) * kEmbedPitch * sizeof(float), st, p));
  MSMD_CHECK_LAUNCH();
  return MSMD_OK;
}

// ------------------------------------------------------------------------------------------- LayerNorm chain
// one warp per 512-wide row; two-pass statistics in registers
template <int D>
__device__ __forceinline__ void ln_row(float (&v)[D / 32], const float* __restrict__ g, const float* __restrict__ b,
                                       int lane) {
  constexpr int NV = D / 32;
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) s += v[i];
  const float mean = warp_sum(s) * (1.0f / D);
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) { const float dlt = v[i] - mean; q = fmaf(dlt, dlt, q); }
  const float rstd = rsqrtf(warp_sum(q) * (1.0f / D) + 1e-5f);
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
template <bool F16>
__device__ __forceinline__ void store_h4(bf16* dst, float a, float b, float c, float d) {
  uint2 u;
  u.x = pack_h<F16>(a, b);
  u.y = pack_h<F16>(c, d);
  *reinterpret_cast<uint2*>(dst) = u;
}
// 4 consecutive 16-bit values -> v[0..3] (ADD: accumulate)
template <bool F16, bool ADD>
__device__ __forceinline__ void load_h4(const bf16* src, float* v) {
  const uint2 u = *reinterpret_cast<const uint2*>(src);
  const float2 a = unpack_h<F16>(u.x), b = unpack_h<F16>(u.y);
  if (ADD) { v[0] += a.x; v[1] += a.y; v[2] += b.x; v[3] += b.y; }
  else { v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y; }
}

// LayerNorm chain of the post-LN layers: out = LN2(LN1(y + resid) + add) (LN3: out = LN(y + resid)).  Inside the replayed
// step y and the residual stream come out of L2 (ncu --cache-control none: 90% L2 hits, 2.5 MB of DRAM traffic), so the
// kernel is bound by instruction issue and load latency, not by HBM.  Hence: a warp owns kLnRows consecutive rows;
// a lane owns two 16-byte chunks of a row (8 + 8 of the 512 features: a quarter of the load instructions of the 8-byte
// version); gamma / beta sit in shared memory (read once per CTA instead of once per row); the raw 16-bit words of the NEXT
// row are in flight while the current one is normalised; statistics are fp32, two-pass, in registers.
template <bool F16>
__device__ __forceinline__ void ln_unpack8(const uint4& u, float* v, bool add) {
  const float2 a = unpack_h<F16>(u.x), b = unpack_h<F16>(u.y), c = unpack_h<F16>(u.z), d = unpack_h<F16>(u.w);
  if (add) { v[0] += a.x; v[1] += a.y; v[2] += b.x; v[3] += b.y; v[4] += c.x; v[5] += c.y; v[6] += d.x; v[7] += d.y; }
  else { v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y; v[4] = c.x; v[5] = c.y; v[6] = d.x; v[7] = d.y; }
}
template <bool F16>
__device__ __forceinline__ uint4 ln_pack8(const float* v) {
  return make_uint4(pack_h<F16>(v[0], v[1]), pack_h<F16>(v[2], v[3]), pack_h<F16>(v[4], v[5]), pack_h<F16>(v[6], v[7]));
}
// normalise the 16 values of this lane (row of 512 over the warp) with gamma / beta from shared memory
__device__ __forceinline__ void ln16(float (&v)[16], const float* __restrict__ sg, const float* __restrict__ sb, int lane) {
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 16; ++i) s += v[i];
  const float mean = warp_sum(s) * (1.0f / 512.0f);
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < 16; ++i) { v[i] -= mean; q = fmaf(v[i], v[i], q); }
  const float rstd = rsqrtf(warp_sum(q) * (1.0f / 512.0f) + 1e-5f);
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const float4 g0 = *reinterpret_cast<const float4*>(sg + h * 256 + lane * 8), g1 = *reinterpret_cast<const float4*>(sg + h * 256 + lane * 8 + 4);
    const float4 b0 = *reinterpret_cast<const float4*>(sb + h * 256 + lane * 8), b1 = *reinterpret_cast<const float4*>(sb + h * 256 + lane * 8 + 4);
    float* w = v + 8 * h;
    w[0] = fmaf(w[0] * rstd, g0.x, b0.x); w[1] = fmaf(w[1] * rstd, g0.y, b0.y); w[2] = fmaf(w[2] * rstd, g0.z, b0.z); w[3] = fmaf(w[3] * rstd, g0.w, b0.w);
    w[4] = fmaf(w[4] * rstd, g1.x, b1.x); w[5] = fmaf(w[5] * rstd, g1.y, b1.y); w[6] = fmaf(w[6] * rstd, g1.z, b1.z); w[7] = fmaf(w[7] * rstd, g1.w, b1.w);
  }
}

template <int D, bool F16, int kLnRows>
__global__ void __launch_bounds__(256) ln_kernel(LnParams p) {
  static_assert(D == 512, "lane layout: two 8-element chunks per lane");
  griddep_launch();
  __shared__ __align__(16) float sgb[4][D];          // g1, b1, g2, b2
  for (int i = threadIdx.x; i < D; i += blockDim.x) {
    sgb[0][i] = p.g1[i]; sgb[1][i] = p.b1[i];
    sgb[2][i] = p.g2 ? p.g2[i] : 0.f; sgb[3][i] = p.b2 ? p.b2[i] : 0.f;
  }
  griddep_wait();
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int row0 = (blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * kLnRows;
  const int c0 = lane * 8, c1 = 256 + lane * 8;
  struct Raw { uint4 y0, y1, r0, r1, a0, a1; };
  auto load = [&](int row, Raw& w) {
    if (row >= p.M) return;
    const bf16* y = p.y + (int64_t)row * D;
    w.y0 = *reinterpret_cast<const uint4*>(y + c0); w.y1 = *reinterpret_cast<const uint4*>(y + c1);
    if (p.resid != nullptr) {
      const bf16* r = p.resid + (int64_t)row * D;
      w.r0 = *reinterpret_cast<const uint4*>(r + c0); w.r1 = *reinterpret_cast<const uint4*>(r + c1);
    }
    const int s = row / p.T, tok = row - s * p.T;
    if (p.add != nullptr && tok > 0) {
      const bf16* a = p.add + ((int64_t)s * (p.T - 1) + (tok - 1)) * D;
      w.a0 = __ldg(reinterpret_cast<const uint4*>(a + c0)); w.a1 = __ldg(reinterpret_cast<const uint4*>(a + c1));
    }
  };
  Raw cur, nxt;
  load(row0, cur);
#pragma unroll
  for (int i = 0; i < kLnRows; ++i) {
    const int row = row0 + i;
    if (i + 1 < kLnRows) load(row + 1, nxt);
    if (row < p.M) {
      const int s = row / p.T, tok = row - s * p.T;
      float v[16];
      ln_unpack8<F16>(cur.y0, v, false); ln_unpack8<F16>(cur.y1, v + 8, false);
      if (p.resid != nullptr) {  // x + sublayer(x): the residual add of the post-LN layer (model.py:874-878)
        ln_unpack8<F16>(cur.r0, v, true); ln_unpack8<F16>(cur.r1, v + 8, true);
      }
      if (!(tok == 0 && p.skip_tok0)) {
        ln16(v, sgb[0], sgb[1], lane);
        if (tok == 0 && p.x0 != nullptr) {
          bf16* o = p.x0 + (int64_t)s * D;
          *reinterpret_cast<uint4*>(o + c0) = ln_pack8<F16>(v); *reinterpret_cast<uint4*>(o + c1) = ln_pack8<F16>(v + 8);
        } else {
          if (p.add != nullptr && tok > 0) {
            // x1 is rounded to 16 bits where the reference's next sub-layer reads it; keep the same rounding point
            ln_unpack8<F16>(cur.a0, v, true); ln_unpack8<F16>(cur.a1, v + 8, true);
            ln16(v, sgb[2], sgb[3], lane);
          }
          bf16* o = p.out + (int64_t)row * D;
          *reinterpret_cast<uint4*>(o + c0) = ln_pack8<F16>(v); *reinterpret_cast<uint4*>(o + c1) = ln_pack8<F16>(v + 8);
        }
      }
    }
    cur = nxt;
  }
}
// Default kernel: one row per warp, 8-byte loads, parameters from global memory (46 registers: high occupancy)
template <int D, bool F16>
__global__ void __launch_bounds__(256) ln_kernel_v1(LnParams p) {
  griddep_launch();
  griddep_wait();
  constexpr int NV = D / 32;
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= p.M) return;
  const int s = row / p.T, tok = row % p.T;
  float v[NV];
  const bf16* y = p.y + (int64_t)row * D;
#pragma unroll
  for (int i = 0; i < NV / 4; ++i) load_h4<F16, false>(y + i * 128 + lane * 4, v + 4 * i);
  if (p.resid != nullptr) {
    const bf16* r = p.resid + (int64_t)row * D;
#pragma unroll
    for (int i = 0; i < NV / 4; ++i) load_h4<F16, true>(r + i * 128 + lane * 4, v + 4 * i);
  }
  if (tok == 0 && p.skip_tok0) return;
  ln_row<D>(v, p.g1, p.b1, lane);
  if (tok == 0 && p.x0 != nullptr) {
#pragma unroll
    for (int i = 0; i < NV / 4; ++i)
      store_h4<F16>(p.x0 + (int64_t)s * D + i * 128 + lane * 4, v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
    return;
  }
  if (p.add != nullptr && tok > 0) {
    const bf16* a = p.add + ((int64_t)s * (p.T - 1) + (tok - 1)) * D;
#pragma unroll
    for (int i = 0; i < NV / 4; ++i) load_h4<F16, true>(a + i * 128 + lane * 4, v + 4 * i);
    ln_row<D>(v, p.g2, p.b2, lane);
  }
  bf16* o = p.out + (int64_t)row * D;
#pragma unroll
  for (int i = 0; i < NV / 4; ++i) store_h4<F16>(o + i * 128 + lane * 4, v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
}
int ln_launch(const LnParams& p, cudaStream_t st) {
  MSMD_REQUIRE(p.d == 512, "ln: only d_model = 512 is instantiated (got %d)", p.d);
  ProfileScope prof(p.add ? "ln1_ln2" : "ln3", st);
  // MSMD_LN_ROWS (A/B): 0 = one row per warp with 8-byte loads (default: measured fastest inside the replayed step, where
  // y and the residual stream come out of L2 and occupancy - 46 registers, 2664 CTAs - hides the load latency);
  // 1 / 4 / 6 = the 16-byte-load kernel with that many rows per warp (6: one wave of 444 CTAs at configuration 3;
  // measured 1.2% SLOWER per step than 0 on the same box, 4 rows 3% slower)
  static const int rows = [] { const char* e = getenv("MSMD_LN_ROWS"); return e ? atoi(e) : 0; }();
  if (rows == 0) {
    MSMD_CHECK_CUDA(launch_pdl(p.fp16 ? ln_kernel_v1<512, true> : ln_kernel_v1<512, false>, dim3(cdiv(p.M, 8)), dim3(256), 0, st, p));
  } else if (rows == 1 || p.M <= 148 * 3 * 8) {
    MSMD_CHECK_CUDA(launch_pdl(p.fp16 ? ln_kernel<512, true, 1> : ln_kernel<512, false, 1>, dim3(cdiv(p.M, 8)), dim3(256), 0, st, p));
  } else if (rows == 4 || p.M < 148 * 3 * 8 * 4) {
    MSMD_CHECK_CUDA(launch_pdl(p.fp16 ? ln_kernel<512, true, 4> : ln_kernel<512, false, 4>, dim3(cdiv(p.M, 8 * 4)), dim3(256), 0, st, p));
  } else {
    MSMD_CHECK_CUDA(launch_pdl(p.fp16 ? ln_kernel<512, true, 6> : ln_kernel<512, false, 6>, dim3(cdiv(p.M, 8 * 6)), dim3(256), 0, st, p));
  }
  MSMD_CHECK_LAUNCH();
  return MSMD_OK;
}

template <int D, bool F16>
__global__ void __launch_bounds__(256) ln_row0_kernel(const bf16* __restrict__ y0, const bf16* __restrict__ resid0,
                                                      const float* __restrict__ g, const float* __restrict__ b,
                                                      bf16* __restrict__ out, bf16* __restrict__ out_c, int S, int T) {
  griddep_launch();
  griddep_wait();
  constexpr int NV = D / 32;
  const int lane = threadIdx.x & 31;
  const int s = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (s >= S) return;
  float v[NV];
#pragma unroll
  for (int i = 0; i < NV / 4; ++i) {
    load_h4<F16, false>(y0 + (int64_t)s * D + i * 128 + lane * 4, v + 4 * i);
    if (resid0 != nullptr) load_h4<F16, true>(resid0 + (int64_t)s * D + i * 128 + lane * 4, v + 4 * i);
  }
  ln_row<D>(v, g, b, lane);
#pragma unroll
  for (int i = 0; i < NV / 4; ++i) {
    if (out) store_h4<F16>(out + (int64_t)s * T * D + i * 128 + lane * 4, v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
    if (out_c) store_h4<F16>(out_c + (int64_t)s * D + i * 128 + lane * 4, v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
  }
}
int ln_row0_launch(const bf16* y0, const bf16* resid0, const float* g, const float* b, bf16* out, bf16* out_c, int S,
                   int T, int d, int fp16, cudaStream_t st) {
  MSMD_REQUIRE(d == 512, "ln_row0: only d_model = 512 is instantiated");
  ProfileScope prof("ln_row0", st);
  MSMD_CHECK_CUDA(launch_pdl(fp16 ? ln_row0_kernel<512, true> : ln_row0_kernel<512, false>, dim3(cdiv(S, 8)), dim3(256), 0, st,
                             y0, resid0, g, b, out, out_c, S, T));
  MSMD_CHECK_LAUNCH();
  return MSMD_OK;
}

// ------------------------------------------------------------------------------------------- row-0 cross attention
// Person token (query row 0) over the Tk memory tokens (nn.MultiheadAttention inside _mha_block): one warp per
// (sequence, head), no shared memory and no barriers.  K: lane j of key group g reads its key's 128-byte head
// slice with 8 x 16-byte loads (the half-used sectors of one load are completed by the next, out of L1); V: lane
// owns 2 of the 64 head dims, so a key's V slice is one coalesced 128-byte warp load, prefetched 28 keys ahead.
// HBM-bound: 2 x Tk x d x 2 B per sequence per layer.
constexpr int kCaBatch = 28;
template <bool F16>
__global__ void __launch_bounds__(128, 3) cross_attn_row0_kernel(const bf16* __restrict__ q0, const bf16* __restrict__ kv,
                                                                 bf16* __restrict__ ctx0, int Tk, int H) {
  griddep_launch();
  griddep_wait();
  constexpr int d = 512;
  const int w = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;   // warp = (sequence, head)
  const int s = w / H, h = w % H;
  const bf16* kbase = kv + (int64_t)s * Tk * 2 * d + h * 64;
  const uint32_t* vbase = reinterpret_cast<const uint32_t*>(kbase + d) + lane;
  const int64_t vstride = d;   // one key row = 2d bf16 = d uint32

  uint32_t vb[2][kCaBatch];
  auto load_v = [&](int b, uint32_t (&dst)[kCaBatch]) {
#pragma unroll
    for (int u = 0; u < kCaBatch; ++u) {
      const int j = b * kCaBatch + u;
      dst[u] = j < Tk ? __ldg(vbase + (int64_t)j * vstride) : 0u;
    }
  };
  load_v(0, vb[0]);

  float q[64];
  {
    const uint4* qp = reinterpret_cast<const uint4*>(q0 + (int64_t)s * d + h * 64);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const uint4 u = __ldg(qp + i);
      const uint32_t ww[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float2 f = unpack_h<F16>(ww[k]);
        q[i * 8 + 2 * k] = f.x;
        q[i * 8 + 2 * k + 1] = f.y;
      }
    }
  }
  float sc[4];
#pragma unroll
  for (int grp = 0; grp < 4; ++grp) {
    const int j = grp * 32 + lane;
    float dot = -INFINITY;
    if (j < Tk) {
      const uint4* kp = reinterpret_cast<const uint4*>(kbase + (int64_t)j * 2 * d);
      uint4 kr[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) kr[i] = __ldg(kp + i);
      float acc = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const uint32_t ww[4] = {kr[i].x, kr[i].y, kr[i].z, kr[i].w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const float2 f = unpack_h<F16>(ww[k]);
          acc = fmaf(q[i * 8 + 2 * k], f.x, acc);
          acc = fmaf(q[i * 8 + 2 * k + 1], f.y, acc);
        }
      }
      dot = acc * 0.125f;
    }
    sc[grp] = dot;
  }
  const float m = warp_max(fmaxf(fmaxf(sc[0], sc[1]), fmaxf(sc[2], sc[3])));
  float l = 0.f;
#pragma unroll
  for (int i = 0; i < 4; ++i) { sc[i] = (sc[i] == -INFINITY) ? 0.f : __expf(sc[i] - m); l += sc[i]; }
  l = warp_sum(l);
  float oa = 0.f, ob = 0.f;
  auto consume = [&](int b, const uint32_t (&src)[kCaBatch]) {
#pragma unroll
    for (int u = 0; u < kCaBatch; ++u) {
      const int j = b * kCaBatch + u;            // compile-time after unrolling: sc[] stays in registers
      const float p = __shfl_sync(0xffffffffu, sc[j >> 5], j & 31);
      const float2 f = unpack_h<F16>(src[u]);
      oa = fmaf(p, f.x, oa);
      ob = fmaf(p, f.y, ob);
    }
  };
  load_v(1, vb[1]); consume(0, vb[0]);
  load_v(2, vb[0]); consume(1, vb[1]);
  load_v(3, vb[1]); consume(2, vb[0]);
  consume(3, vb[1]);
  const float inv = 1.0f / l;
  *reinterpret_cast<uint32_t*>(ctx0 + (int64_t)s * d + h * 64 + 2 * lane) = pack_h<F16>(oa * inv, ob * inv);
}
int cross_attn_row0_launch(const bf16* q0, const bf16* kv, bf16* ctx0, int S, int Tk, int H, int fp16, cudaStream_t st) {
  MSMD_REQUIRE(Tk <= 4 * kCaBatch && H == 8, "cross_attn_row0: built for 8 heads x 64 and <= %d memory tokens (got %d, %d)",
               4 * kCaBatch, H, Tk);
  ProfileScope prof("cross_attn_row0", st);
  MSMD_CHECK_CUDA(launch_pdl(fp16 ? cross_attn_row0_kernel<true> : cross_attn_row0_kernel<false>, dim3(S * H / 4), dim3(128), 0, st,
                             q0, kv, ctx0, Tk, H));
  MSMD_CHECK_LAUNCH();
  return MSMD_OK;
}

// ------------------------------------------------------------------------------------------- sampler update
// Philox4x32-10 + Box-Muller for the in-kernel noise path (z == null); keyed by (seed, t, element)
__device__ __forceinline__ float philox_normal(unsigned long long seed, uint32_t t, uint32_t idx) {
  uint32_t c0 = idx, c1 = t, c2 = 0x9E3779B9u, c3 = 0xBB67AE85u;
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    c0 = hi1 ^ c1 ^ k0; c1 = lo1; c2 = hi0 ^ c3 ^ k1; c3 = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  const float u1 = ((c0 >> 8) + 1) * (1.0f / 16777216.0f);
  const float u2 = (c1 >> 8) * (1.0f / 16777216.0f);
  return sqrtf(-2.0f * __logf(u1)) * __cosf(6.283185307179586f * u2);
}

// model.py:964-995: dynamic + sum_b alpha_b * static_b (face dims) / sum_b static_b (last 3 dims, unweighted)
__device__ __forceinline__ void split_target(const float* dec, const float* stat, int T, int Lp, int dm, int nb, int ldd,
                                             int s, int l, int c, float& dyn, float& sta) {
  const float* row = dec + ((int64_t)s * T + 1 + Lp + l) * ldd;
  const float* st = stat + (int64_t)s * nb * dm;
  dyn = row[c];
  const bool face = c < dm - 3;
  float v = 0.f;
  for (int b = 0; b < nb; ++b) v += (face ? row[dm + b] : 1.0f) * st[b * dm + c];
  sta = v;
}

// The parameter block lives in device memory (msmd_model::d_up, rewritten by every msmd_sample_window call with a
// stream-ordered copy): the captured step graph never bakes a caller pointer or scalar, so one instantiated graph
// serves every window / call of the same shape.
__global__ void __launch_bounds__(256) update_kernel(const UpdateParams* __restrict__ pp) {
  griddep_launch();
  griddep_wait();
  // the parameter block is read through shared memory: as a local copy of *pp its ~30 fields were re-fetched from global
  // memory (generic loads) all over the loop, one more dependent latency in front of every data load
  __shared__ __align__(16) unsigned char p_raw[sizeof(UpdateParams)];
  static_assert(sizeof(UpdateParams) % 4 == 0, "UpdateParams is copied in 32-bit words");
  for (int i = threadIdx.x; i < (int)(sizeof(UpdateParams) / 4); i += blockDim.x)
    reinterpret_cast<uint32_t*>(p_raw)[i] = reinterpret_cast<const uint32_t*>(pp)[i];
  __syncthreads();
  const UpdateParams& p = *reinterpret_cast<const UpdateParams*>(p_raw);
  const int64_t n_el = (int64_t)p.NX * p.L * p.dm;
  const int t = p.steps[0];
  float sigma, c0, c1, c2 = 0.f, ha = 0.f, hb = 0.f;
  int t_next = t - 1, ord = p.t_start - t;
  if (p.sched != nullptr) {   // respaced schedule: host-computed coefficients of x_s = c0 x_t + c1 out + c2 h_p + sigma z
    const SchedStep e = p.sched[t];
    c0 = e.c0; c1 = e.c1; sigma = e.sigma; c2 = e.c2; ha = e.a; hb = e.b; t_next = e.next; ord = e.ord;
  } else {
    // model.py:383-386, :421-428 - 0-dim fp32 tensor arithmetic, same operation order
    const float alpha = p.alphas[t], ab = p.alpha_bars[t], abp = p.alpha_bars[t - 1];
    sigma = p.sig_flex[t] * p.flexibility + p.sig_inflex[t] * (1.0f - p.flexibility);
    if (p.target_noise) {
      c0 = 1.0f / sqrtf(alpha);
      c1 = (1.0f - alpha) / sqrtf(1.0f - ab);
    } else {
      c0 = (1.0f - abp) * sqrtf(alpha) / (1.0f - ab);
      c1 = (1.0f - alpha) * sqrtf(abp) / (1.0f - ab);
    }
  }
  // loop-invariant fields in registers: the stores below go through generic pointers that the compiler must assume may
  // alias the shared-memory parameter block, so every p.field in the loop was re-read after each store
  struct Loc {
    const float *dec, *stat, *z, *thr; float *x, *traj, *tgt_dyn, *cum_static, *alpha_traj, *hist; const int* overflow;
    const long long* keys;
    float scale0, scale1; unsigned long long seed; long long noise_offset;
    int NX, E, T, L, Lp, dm, nb, ldd, cfg_independent, target_noise;
  };
  // target_noise here selects the posterior's form x_{t-1} = c0 (x_t - c1 eps_hat); a respaced step is affine in both
  // targets
  const Loc q = {p.dec, p.stat, p.z, p.thr, p.x, p.traj, p.tgt_dyn, p.cum_static, p.alpha_traj, p.hist, p.overflow,
                 p.noise_keys,
                 p.scale0, p.scale1, p.seed, p.noise_offset,
                 p.NX, p.E, p.T, p.L, p.Lp, p.dm, p.nb, p.ldd, p.cfg_independent, p.target_noise && p.sched == nullptr};
  const bool sep = q.tgt_dyn != nullptr || q.cum_static != nullptr;
  // warp = one (clip, frame) row of dm codes, lane = column c (+32, +64): no 64-bit index arithmetic per element (three
  // int64 divisions per element made this kernel instruction-bound: 600 instructions per element, 23 us per step)
  const int lane = threadIdx.x & 31;
  const int rows = q.NX * q.L;
  for (int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); row < rows; row += gridDim.x * (blockDim.x >> 5)) {
    const int n = row / q.L, l = row - n * q.L;
    // per-row invariants of the (<= 3) guidance entries: decoder row, static-basis block, threshold, mixing weights
    const float* rowp[3];
    const float* stp[3];
    float thv[3], al[3][4];
#pragma unroll
    for (int e = 0; e < 3; ++e) {
      const int sq = (e < q.E ? e : 0) * q.NX + n;
      rowp[e] = q.dec + ((int64_t)sq * q.T + 1 + q.Lp + l) * q.ldd;
      stp[e] = q.stat + (int64_t)sq * q.nb * q.dm;
      thv[e] = q.thr ? q.thr[sq] : 0.f;
#pragma unroll
      for (int b = 0; b < 4; ++b) al[e][b] = b < q.nb ? rowp[e][q.dm + b] : 0.f;
    }
    // Philox key of the row: element index (global clip id * L + l) * dm + c under the clip's seed.  Without per-clip keys
    // the global clip id is noise_clip_offset + n, i.e. the index is i + noise_offset (32-bit wrap-around either way)
    unsigned long long nseed = q.seed;
    long long nbase = (long long)row * q.dm + q.noise_offset;
    if (q.keys != nullptr) {
      nseed = (unsigned long long)q.keys[2 * n];
      nbase = (long long)l * q.dm + q.keys[2 * n + 1] * q.L * q.dm;
    }
   for (int c = lane; c < q.dm; c += 32) {
    const int64_t i = (int64_t)row * q.dm + c;
    const bool face = c < q.dm - 3;
    // CFG combine (model.py:404-417); results[0] is updated in place through a view, so 'independent'
    // subtracts the running target (SURVEY App. C-4).  The same recursion runs on the dynamic / static parts
    // (model.py:603-626) when the separate outputs are requested.
    float tgt = 0.f, prev = 0.f, td = 0.f, pd = 0.f, ts = 0.f, psv = 0.f;
#pragma unroll
    for (int e = 0; e < 3; ++e) {
      if (e >= q.E) break;
      // split_target() with the row's pointers / mixing weights held in registers (same operation order)
      const float dyn = rowp[e][c];
      float sta = 0.f;
      if (q.nb <= 4) {
#pragma unroll
        for (int b = 0; b < 4; ++b)
          if (b < q.nb) sta += (face ? al[e][b] : 1.0f) * stp[e][b * q.dm + c];
      } else {
        for (int b = 0; b < q.nb; ++b) sta += (face ? rowp[e][q.dm + b] : 1.0f) * stp[e][b * q.dm + c];
      }
      float r = dyn + sta;
      if (q.thr) { const float th = thv[e]; r = fminf(fmaxf(r, -th), th); }
      if (e == 0) {
        tgt = r; td = dyn; ts = sta;
      } else {
        const float sc = (e == 1) ? q.scale0 : q.scale1;
        const bool run = q.cfg_independent || e == 1;
        tgt = tgt + sc * (r - (run ? tgt : prev));
        if (sep) { td = td + sc * (dyn - (run ? td : pd)); ts = ts + sc * (sta - (run ? ts : psv)); }
      }
      prev = r; pd = dyn; psv = sta;
    }
    float zt = 0.f;
    if (t_next > 0) zt = q.z ? q.z[(int64_t)t * n_el + i] : philox_normal(nseed, (uint32_t)t, (uint32_t)(nbase + c));
    const float xo = q.x[i];
    // DPM-Solver++(2M) steps read the previous step's data prediction and leave their own for the next step; DDIM
    // steps and the default loop keep their expression (c2 = b = 0, uniform over the grid)
    float xn;
    if (c2 != 0.f) xn = c0 * xo + c1 * tgt + c2 * q.hist[i] + sigma * zt;
    else xn = q.target_noise ? (c0 * (xo - c1 * tgt) + sigma * zt) : (c0 * xo + c1 * tgt + sigma * zt);
    if (hb != 0.f) q.hist[i] = ha * xo + hb * tgt;
    // fp32-grade steps: an activation left the fp16 range of the operand split -> poison the state instead of
    // returning a silently wrong sample (the host reports it at the next call, without synchronising this one)
    if (q.overflow != nullptr && *q.overflow != 0) xn = __int_as_float(0x7fc00000);
    q.x[i] = xn;
    if (q.traj) q.traj[(int64_t)t_next * n_el + i] = xn;
    if (q.tgt_dyn) q.tgt_dyn[i] = td;
    if (q.cum_static) q.cum_static[i] += c1 * ts;
    if (q.alpha_traj && c < q.nb) {   // alphas: columns dm..dm+nb-1 of the decoder output, same CFG recursion
      float ta = 0.f, pa = 0.f;
      for (int e = 0; e < q.E; ++e) {
        const float a = q.dec[((int64_t)(e * q.NX + n) * q.T + 1 + q.Lp + l) * q.ldd + q.dm + c];
        if (e == 0) ta = a;
        else ta = ta + ((e == 1) ? q.scale0 : q.scale1) * (a - ((q.cfg_independent || e == 1) ? ta : pa));
        pa = a;
      }
      q.alpha_traj[(((int64_t)ord * q.NX + n) * q.L + l) * q.nb + c] = ta;
    }
   }
  }
  // step index t -> t_next for the next step, by the LAST block to finish (every block has read t by then): the separate
  // one-thread-block "advance" launch of round 1 is gone
  if (p.done != nullptr) {
    __shared__ bool last;
    __syncthreads();
    if (threadIdx.x == 0) {
      __threadfence();
      last = atomicAdd(p.done, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (last) {
      for (int i = threadIdx.x; i < p.S; i += blockDim.x) p.steps_rw[i] = t_next;
      if (threadIdx.x == 0) *p.done = 0u;
    }
  }
}

// Dynamic thresholding (model.py:396-402): one CTA per sequence; |x0_hat| of the L motion rows in shared memory,
// exact k-th order statistics by 4-pass radix select on the float bit patterns, linear interpolation like
// torch.quantile(..., interpolation='linear').
__global__ void __launch_bounds__(1024) threshold_kernel(const float* __restrict__ dec, const float* __restrict__ stat,
                                                         float* __restrict__ thr, int T, int L, int Lp, int dm, int nb,
                                                         int ldd, float ratio, float lo, float hi) {
  extern __shared__ uint32_t keys[];   // [L*dm] then hist[256], sel[4]
  const int n = L * dm;
  uint32_t* hist = keys + n;
  uint32_t* sel = hist + 256;
  const int s = blockIdx.x, tid = threadIdx.x;
  for (int i = tid; i < n; i += blockDim.x) {
    float dyn, sta;
    split_target(dec, stat, T, Lp, dm, nb, ldd, s, i / dm, i % dm, dyn, sta);
    keys[i] = __float_as_uint(fabsf(dyn + sta));
  }
  const float pos = ratio * (float)(n - 1);
  const int k_lo = (int)floorf(pos), k_hi = (int)ceilf(pos);
  float v[2];
  for (int which = 0; which < 2; ++which) {
    int k = which == 0 ? k_lo : k_hi;
    uint32_t prefix = 0, mask = 0;
    for (int pass = 3; pass >= 0; --pass) {
      for (int i = tid; i < 256; i += blockDim.x) hist[i] = 0;
      __syncthreads();
      for (int i = tid; i < n; i += blockDim.x) {
        const uint32_t key = keys[i];
        if ((key & mask) == prefix) atomicAdd(&hist[(key >> (8 * pass)) & 255u], 1u);
      }
      __syncthreads();
      if (tid == 0) {
        uint32_t cum = 0, b = 0;
        for (; b < 256; ++b) {
          if (cum + hist[b] > (uint32_t)k) break;
          cum += hist[b];
        }
        sel[0] = b; sel[1] = cum;
      }
      __syncthreads();
      prefix |= sel[0] << (8 * pass);
      mask |= 255u << (8 * pass);
      k -= (int)sel[1];
      __syncthreads();
    }
    v[which] = __uint_as_float(prefix);
  }
  if (tid == 0) {
    const float w = pos - (float)k_lo;
    const float q = v[0] + w * (v[1] - v[0]);     // torch.lerp form
    thr[s] = fminf(fmaxf(q, lo), hi);
  }
}
int threshold_launch(const float* dec, const float* stat, float* thr, int S, int T, int L, int Lp, int dm, int nb, int ldd,
                     float ratio, float lo, float hi, cudaStream_t st) {
  MSMD_REQUIRE(ratio >= 0.f && ratio <= 1.f, "quantile() q values must be in the range [0, 1] (got %f)", ratio);
  const size_t smem = ((size_t)L * dm + 256 + 4) * sizeof(uint32_t);
  MSMD_REQUIRE(smem <= 48 * 1024, "threshold: %d values per sequence exceed the shared-memory tile", L * dm);
  threshold_kernel<<<S, 1024, smem, st>>>(dec, stat, thr, T, L, Lp, dm, nb, ldd, ratio, lo, hi);
  MSMD_CHECK_LAUNCH();
  return MSMD_OK;
}

__global__ void update_params_set_kernel(UpdateParams* dst, const UpdateParams src) { *dst = src; }
int update_params_set(UpdateParams* d_dst, const UpdateParams& p, cudaStream_t st) {
  update_params_set_kernel<<<1, 1, 0, st>>>(d_dst, p);   // by-value kernel argument: stream-ordered, no host staging buffer to keep alive
  MSMD_CHECK_LAUNCH();
  return MSMD_OK;
}
int update_launch(const UpdateParams* d_p, int NX, int L, int dm, cudaStream_t st) {
  (void)dm;
  ProfileScope prof("update", st);
  // warp per row, ONE wave (2 CTAs of 123 registers per SM): every CTA starts with a chain of dependent scalar loads
  // (parameter block -> step index -> schedule coefficients, ~2 us); the 4-wave grid of round 1 paid it four times
  MSMD_CHECK_CUDA(launch_pdl(update_kernel, dim3(std::min(cdiv(NX * L, 8), kNumSMs * 2)), dim3(256), 0, st, d_p));
  MSMD_CHECK_LAUNCH();
  return MSMD_OK;
}

// 512 entries = 18 KB of kernel parameters (the limit is 32 KB): one launch for any schedule of the 500-step models
constexpr int kSchedChunk = 512;
struct SchedChunk {
  int n;
  SchedStep e[kSchedChunk];
};
static_assert(sizeof(SchedChunk) <= 32764, "sched_table_set: a chunk must fit the kernel-parameter limit");
__global__ void sched_table_set_kernel(SchedStep* table, const SchedChunk c) {
  for (int i = threadIdx.x; i < c.n; i += blockDim.x) table[c.e[i].t] = c.e[i];
}
int sched_table_set(SchedStep* table, const SchedStep* h, int n, cudaStream_t st) {
  for (int a = 0; a < n; a += kSchedChunk) {
    SchedChunk c;
    c.n = std::min(kSchedChunk, n - a);
    memcpy(c.e, h + a, c.n * sizeof(SchedStep));
    sched_table_set_kernel<<<1, 256, 0, st>>>(table, c);
    MSMD_CHECK_LAUNCH();
  }
  return MSMD_OK;
}

__global__ void steps_set_kernel(int* steps, int S, int v) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < S) steps[i] = v;
}
int steps_set(int* steps, int S, int value, cudaStream_t st) {
  steps_set_kernel<<<cdiv(S, 256), 256, 0, st>>>(steps, S, value);
  MSMD_CHECK_LAUNCH();
  return MSMD_OK;
}
__global__ void mix_static_kernel(const float* __restrict__ dec, const float* __restrict__ stat, float* __restrict__ out,
                                  int S, int T, int dm, int nb, int ldd) {
  const int64_t n_el = (int64_t)S * (T - 1) * dm;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_el; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % dm);
    const int tok = (int)((i / dm) % (T - 1));
    const int s = (int)(i / ((int64_t)dm * (T - 1)));
    const float* row = dec + ((int64_t)s * T + 1 + tok) * ldd;
    float v = row[c];
    const bool face = c < dm - 3;
    for (int b = 0; b < nb; ++b) v += (face ? row[dm + b] : 1.0f) * stat[((int64_t)s * nb + b) * dm + c];
    out[i] = v;
  }
}
int mix_static_launch(const float* dec, const float* stat, float* out, int S, int T, int dm, int nb, int ldd,
                      cudaStream_t st) {
  const int64_t n = (int64_t)S * (T - 1) * dm;
  mix_static_kernel<<<(int)std::min<int64_t>(cdiv(n, 256), kNumSMs * 8), 256, 0, st>>>(dec, stat, out, S, T, dm, nb, ldd);
  MSMD_CHECK_LAUNCH();
  return MSMD_OK;
}


// keep_separate=True outputs of DenoisingNetwork_MSMD.forward (model.py:964-983): the dynamic features, the raw
// static-basis outputs tiled over the Lp+L rows, and the alphas - no mixing.
__global__ void split_parts_kernel(const float* __restrict__ dec, const float* __restrict__ stat, float* __restrict__ dyn,
                                   float* __restrict__ sta, float* __restrict__ alphas, int S, int T, int dm, int nb, int ldd) {
  const int64_t rows = (int64_t)S * (T - 1);
  const int per_row = dm + nb * dm + nb;
  const int64_t n = rows * per_row;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / per_row;
    const int k = (int)(i % per_row);
    const int s = (int)(r / (T - 1)), tok = (int)(r % (T - 1));
    const float* row = dec + ((int64_t)s * T + 1 + tok) * ldd;
    if (k < dm) dyn[r * dm + k] = row[k];
    else if (k < dm + nb * dm) sta[r * nb * dm + (k - dm)] = stat[(int64_t)s * nb * dm + (k - dm)];
    else alphas[r * nb + (k - dm - nb * dm)] = row[dm + (k - dm - nb * dm)];
  }
}
int split_parts_launch(const float* dec, const float* stat, float* dyn, float* sta, float* alphas, int S, int T, int dm,
                       int nb, int ldd, cudaStream_t st) {
  const int64_t n = (int64_t)S * (T - 1) * (dm + nb * dm + nb);
  split_parts_kernel<<<(int)std::min<int64_t>(cdiv(n, 256), kNumSMs * 8), 256, 0, st>>>(dec, stat, dyn, sta, alphas, S, T, dm,
                                                                                        nb, ldd);
  MSMD_CHECK_LAUNCH();
  return MSMD_OK;
}

}  // namespace msmd
