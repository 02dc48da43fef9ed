// Person-token (row 0) cross-attention block of a decoder layer as ONE kernel (nn.TransformerDecoderLayer._mha_block +
// norm2 for the query row that sees the whole memory, model.py:879-883 / :951-958):
//
//     x[s, 0, :] = LayerNorm2( x0c[s] + Wco . attn_h( Wq0 . x0c[s] + bq0 ; K_s, V_s ) + bco )
//
// It replaces four launches (q-projection GEMM, warp-per-head attention, out-projection GEMM, LayerNorm) that cost
// ~31 us per layer on the critical path for S rows of work (S = sequences, 192 at config 3; 3 in the batch-1 latency
// regime, where the three saved launches per layer are 20% of the step).
//
// One thread-block CLUSTER of 8 CTAs per group of <= 16 sequences, CTA rank = attention head h:
//   phase 0  stage this head's weight slices in shared memory once per CTA: Wq0 rows [64h, 64h+64) (64 KB) and the
//            K-slice Wco[:, 64h:64h+64) (64 KB); L2-prefetch the head's K / V cache lines of the group's sequences;
//   phase 1  q_h = Wq0_h . x0c + b      [64 x 512] x [512 x n]   warp-level mma.sync m16n8k16 (the sequences are the
//            N columns, ldmatrix'd weight rows the A operand): 16 warps = 4 output tiles x 4 K quarters, summed in a
//            fixed order.  (The CUDA-core version of this phase was shared-memory-bandwidth bound: 5500 cycles per 7
//            sequences; a tcgen05 tile would idle 120 of its 128 rows.)
//   phase 2  attention of head h: warp w = keys [8w, 8w+8) of every sequence, four sequences' K / V rows in flight
//            per warp (HBM / L2-bound: the K/V cache is the only large read of the kernel)
//   phase 3  partial out-projection po = Wco[:, h-slice] . ctx_h   [512 x 64] x [64 x n], mma.sync again
//   phase 4  distributed-shared-memory reduction of the 8 partial projections: CTA h finishes the rows of sequences h and
//            h + 8 of the group (thread = column): sums the 8 partials over DSMEM, adds residual + bias, block LayerNorm.
// Two cluster barriers per group.  16-bit storage format (bf16 / fp16) is a template parameter like everywhere else.
// Every sequence is a column of the MMAs and a private slice of the attention partials: its arithmetic does not depend
// on which other sequences share the cluster, so a clip's codes are bit-identical whatever batch it is sampled in.
#include "denoiser_kernels.cuh"
#include "profile.cuh"
#include <cuda_fp16.h>

namespace msmd {
namespace {

constexpr int kThreads = 512, kNB = 16, kD = 512, kDh = 64, kHeads = 8;
constexpr int kParts = 14, kPartKeys = 8;   // the memory keys are ALWAYS cut into 14 parts of 8 (Tk <= 112)
constexpr int kWqPitch = kD + 8;        // halfs per staged Wq0 row (1040 B: 16-byte aligned, rows 4 banks apart: ldmatrix conflict-free)
constexpr int kWoPitch = kDh + 8;       // halfs per staged Wco row slice (144 B, same stagger)
constexpr int kXPitch = kD + 8;         // halfs per x0c row (B operand of the q projection)
constexpr int kCPitch = kDh + 8;        // halfs per ctx row (B operand of the out-projection)
constexpr int kPoPitch = kD + 4;        // floats per partial-projection row
constexpr int kPartFloats = 66;         // max, sum, o[64]
constexpr int kOffWq = 0;
constexpr int kOffWo = kOffWq + kDh * kWqPitch * 2;
constexpr int kOffXs = kOffWo + kD * kWoPitch * 2;
constexpr int kOffQs = kOffXs + kNB * kXPitch * 2;
constexpr int kOffCs = kOffQs + kNB * kDh * 4;
constexpr int kOffPo = kOffCs + kNB * kCPitch * 2;
// one buffer, three lives per group: K-quarter partials of the q projection [4][64][16], attention partials
// [16][14][66], partial out-projection [16][516] (each is dead before the next is written)
constexpr int kPoBytes = kNB * kParts * kPartFloats * 4;
constexpr int kOffSt = kOffPo + kPoBytes;
constexpr int kSmem = kOffSt + 2 * 32 * 4;      // LayerNorm block-reduction scratch: [2 rows][sum(16 warps) | sq(16 warps)]
constexpr int kMaxGroup = kNB;          // sequences per cluster pass = two 8-column MMA tiles
static_assert(kNB * kPoPitch * 4 <= kPoBytes && 4 * kDh * kNB * 4 <= kPoBytes, "po / q-partial views must fit the shared buffer");
static_assert(kOffWo % 16 == 0 && kOffXs % 16 == 0 && kOffQs % 16 == 0 && kOffCs % 16 == 0 && kOffPo % 16 == 0 && kOffSt % 16 == 0, "alignment");
static_assert(kSmem <= 227 * 1024, "row0_fused shared memory");

struct Row0Params {
  const bf16* x0c;     // [S, 512]   LayerNorm1 output of the person rows
  const bf16* Wq;      // [512, 512] cross-attention query projection
  const float* bq;
  const bf16* kv;      // [S, Tk, 1024] memory K | V projections (per-window cache)
  const bf16* Wo;      // [512, 512] cross-attention out-projection
  const float* bo;
  const float* g;      // norm2
  const float* be;
  bf16* x;             // [S, T, 512] residual stream: row 0 of every sequence is written
  int S, T, Tk;
  unsigned long long* trace;   // -DMSMD_ROW0_TRACE builds: clock64 stamps of CTA 0 at the phase boundaries
};

template <bool F16>
__device__ __forceinline__ float2 up2(uint32_t w) {
  if constexpr (F16) return __half22float2(*reinterpret_cast<const __half2*>(&w));
  else return make_float2(__uint_as_float(w << 16), __uint_as_float(w & 0xffff0000u));
}
template <bool F16>
__device__ __forceinline__ uint32_t pk2(float a, float b) {
  if constexpr (F16) {
    __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
  } else {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
  }
}
template <bool F16>
__device__ __forceinline__ void up8(const uint4& u, float* f) {
  const float2 a = up2<F16>(u.x), b = up2<F16>(u.y), c = up2<F16>(u.z), d = up2<F16>(u.w);
  f[0] = a.x; f[1] = a.y; f[2] = b.x; f[3] = b.y; f[4] = c.x; f[5] = c.y; f[6] = d.x; f[7] = d.y;
}
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
__device__ __forceinline__ void r0_stamp(unsigned long long* tr, int ev) {
#ifdef MSMD_ROW0_TRACE
  if (tr != nullptr && blockIdx.x == 0 && threadIdx.x == 0) tr[ev] = clock64();
#endif
}
__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem)), "l"(gmem)
               : "memory");
}
__device__ __forceinline__ uint32_t ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_barrier() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// address of `p` (a shared-memory location of this CTA) in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t remote_addr(const void* p, uint32_t rank) {
  uint32_t a = (uint32_t)__cvta_generic_to_shared(p), r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(rank));
  return r;
}
__device__ __forceinline__ float2 ld_remote_f2(uint32_t addr) {
  float2 v;
  asm volatile("ld.shared::cluster.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ float ld_remote_f(uint32_t addr) {
  float v;
  asm volatile("ld.shared::cluster.f32 %0, [%1];" : "=f"(v) : "r"(addr) : "memory");
  return v;
}

__device__ __forceinline__ void ldmatrix_x4(uint32_t (&r)[4], const void* smem_row) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"((uint32_t)__cvta_generic_to_shared(smem_row)));
}
// D (16x8, fp32) += A (16x16, row-major) . B (16x8, K-major per column), 16-bit operands in the storage format
template <bool F16>
__device__ __forceinline__ void mma16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  if constexpr (F16)
    asm("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3]) : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
  else
    asm("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3]) : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

template <bool F16>
__global__ void __cluster_dims__(kHeads, 1, 1) __launch_bounds__(kThreads, 1) row0_fused_kernel(const Row0Params p) {
  extern __shared__ __align__(16) uint8_t sm[];
  r0_stamp(p.trace, 0);
  bf16* wq = reinterpret_cast<bf16*>(sm + kOffWq);
  bf16* wo = reinterpret_cast<bf16*>(sm + kOffWo);
  bf16* xs = reinterpret_cast<bf16*>(sm + kOffXs);
  float* qs = reinterpret_cast<float*>(sm + kOffQs);
  bf16* cs = reinterpret_cast<bf16*>(sm + kOffCs);   // ctx_h of the group, 16-bit (the format every attention output is stored in)
  float* po = reinterpret_cast<float*>(sm + kOffPo);
  float* st = reinterpret_cast<float*>(sm + kOffSt);   // [2][32]
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int gid = lane >> 2, tig = lane & 3;           // mma.sync fragment coordinates
  const int h = (int)ctarank();
  const int cid = blockIdx.x / kHeads, ncl = gridDim.x / kHeads;
  const int s_begin = (int)(((int64_t)p.S * cid) / ncl), s_end = (int)(((int64_t)p.S * (cid + 1)) / ncl);

  // ---- phase 0a: weight slices, asynchronously (cp.async: all 16 chunks of a thread in flight at once; they are
  // only needed by phase 1 / phase 3).
#pragma unroll
  for (int u = 0; u < kDh * (kD / 8) / kThreads; ++u) {        // Wq0 rows 64h..64h+63, 64 x 16-byte chunks each
    const int i = tid + u * kThreads, r = i >> 6, c = i & 63;
    cp_async16(wq + r * kWqPitch + c * 8, p.Wq + (int64_t)(h * kDh + r) * kD + c * 8);
  }
  asm volatile("cp.async.commit_group;" ::: "memory");
#pragma unroll
  for (int u = 0; u < kD * (kDh / 8) / kThreads; ++u) {        // Wco[:, 64h..64h+63]: 512 rows x 8 chunks
    const int i = tid + u * kThreads, r = i >> 3, c = i & 7;
    cp_async16(wo + r * kWoPitch + c * 8, p.Wo + (int64_t)r * kD + h * kDh + c * 8);
  }
  asm volatile("cp.async.commit_group;" ::: "memory");

  for (int s0 = s_begin; s0 < s_end; s0 += kMaxGroup) {
    const int n = min(kMaxGroup, s_end - s0);
    const int ntiles = (n + 7) >> 3;           // 8-sequence MMA column tiles in use
    // ---- phase 0b: x0c rows of the group (zero-padded to kNB) + L2 prefetch of this head's K / V lines
    for (int i = tid; i < kNB * (kD / 8); i += kThreads) {
      const int s = i >> 6, c = i & 63;
      uint4 v = make_uint4(0, 0, 0, 0);
      if (s < n) v = *reinterpret_cast<const uint4*>(p.x0c + (int64_t)(s0 + s) * kD + c * 8);
      *reinterpret_cast<uint4*>(xs + s * kXPitch + c * 8) = v;
    }
    for (int i = tid; i < n * p.Tk * 2; i += kThreads) {
      const int s = i / (p.Tk * 2), r = i % (p.Tk * 2);
      const bf16* line = p.kv + ((int64_t)(s0 + s) * p.Tk + (r >> 1)) * (2 * kD) + (r & 1) * kD + h * kDh;
      asm volatile("prefetch.global.L2 [%0];" ::"l"(line));
    }
    asm volatile("cp.async.wait_group 1;" ::: "memory");     // Wq0 slice has landed (Wco may still be in flight)
    __syncthreads();
    r0_stamp(p.trace, 1);

    const int part = warp, base = part * kPartKeys;       // attention: warp w = keys [8w, 8w+8) of every sequence (w < kParts)
    const int nk = max(0, min(kPartKeys, p.Tk - base));   // keys of this part
    const int j = lane >> 2, qd = lane & 3;
    const bool valid = j < nk;
    // two register buffers of two sequences each: the loads of the NEXT pair of sequences are in flight while the
    // current pair is scored (with one 4-sequence buffer the phase paid a full memory latency per chunk: 24.8K cycles
    // for 13 sequences at configuration 3)
    struct KV { uint4 ka[2], kb[2]; uint32_t vr[2][8]; };
    auto load2 = [&](KV& r, int c0) {
#pragma unroll
      for (int u2 = 0; u2 < 2; ++u2) {
        if (c0 + u2 < n) {
          const bf16* kbase = p.kv + ((int64_t)(s0 + c0 + u2) * p.Tk + base) * (2 * kD) + h * kDh;
          r.ka[u2] = r.kb[u2] = make_uint4(0, 0, 0, 0);
          if (valid) {
            const uint4* kp = reinterpret_cast<const uint4*>(kbase + (int64_t)j * (2 * kD) + qd * 16);
            r.ka[u2] = __ldg(kp);
            r.kb[u2] = __ldg(kp + 1);
          }
          const uint32_t* vbase = reinterpret_cast<const uint32_t*>(kbase + kD) + lane;
#pragma unroll
          for (int u = 0; u < 8; ++u) r.vr[u2][u] = u < nk ? __ldg(vbase + (int64_t)u * kD) : 0u;
        }
      }
    };
    KV bufA, bufB;
    // the first pair of sequences is requested NOW: K / V do not depend on q, so this latency hides under the q projection
    if (warp < kParts) load2(bufA, 0);

    // ---- phase 1: q_h[s][o] = bq[64h+o] + sum_k Wq0[64h+o][k] x0c[s][k].  Warp = (output tile mt of 16, K quarter kq);
    // the four K-quarter partials of every (o, s) are summed below in a fixed order.
    {
      const int mt = warp & 3, kq = warp >> 2;
      float acc[2][4];
#pragma unroll
      for (int nt = 0; nt < 2; ++nt)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[nt][j] = 0.f;
      const bf16* arow = wq + (16 * mt + (lane & 7) + ((lane >> 3) & 1) * 8) * kWqPitch + (lane >> 4) * 8 + 128 * kq;
      const bf16* brow = xs + gid * kXPitch + 128 * kq + tig * 2;
#pragma unroll
      for (int ks = 0; ks < 8; ++ks) {
        uint32_t a[4];
        ldmatrix_x4(a, arow + 16 * ks);
#pragma unroll
        for (int nt = 0; nt < 2; ++nt) {
          if (nt < ntiles) {
            const uint32_t b0 = *reinterpret_cast<const uint32_t*>(brow + nt * 8 * kXPitch + 16 * ks);
            const uint32_t b1 = *reinterpret_cast<const uint32_t*>(brow + nt * 8 * kXPitch + 16 * ks + 8);
            mma16816<F16>(acc[nt], a, b0, b1);
          }
        }
      }
      float* qpart = po + kq * (kDh * kNB);         // [kq][o][seq]
#pragma unroll
      for (int nt = 0; nt < 2; ++nt) {
        if (nt < ntiles) {
          *reinterpret_cast<float2*>(qpart + (16 * mt + gid) * kNB + 8 * nt + 2 * tig) = make_float2(acc[nt][0], acc[nt][1]);
          *reinterpret_cast<float2*>(qpart + (16 * mt + gid + 8) * kNB + 8 * nt + 2 * tig) = make_float2(acc[nt][2], acc[nt][3]);
        }
      }
    }
    __syncthreads();
    for (int i = tid; i < kDh * kNB; i += kThreads) {
      const int o = i >> 4, s = i & 15;
      if (s < 8 * ntiles) {
        float v = po[0 * (kDh * kNB) + i];
        v += po[1 * (kDh * kNB) + i];
        v += po[2 * (kDh * kNB) + i];
        v += po[3 * (kDh * kNB) + i];
        qs[s * kDh + o] = v + __ldg(p.bq + h * kDh + o);
      }
    }
    __syncthreads();

    // ---- phase 2: attention of head h.  The Tk <= 112 keys are ALWAYS cut into 14 parts of 8 keys, warp w = part w of
    // every sequence of the group: each part yields a partial (max, sum, P V) and the parts are merged in a fixed
    // order below - the arithmetic of a sequence does not depend on how many sequences share the cluster.  Lane
    // (j, qd) = (lane / 4, lane % 4) scores 16 of the 64 head dims of key 8w + j (two 16-byte loads; the 4-lane sums are
    // two shuffles); every lane owns two of the 64 head dims for P V (one coalesced 128-byte warp load per key).
    r0_stamp(p.trace, 2);
    float* parts = po;                              // [seq][kParts][66]: m, l, o(64)
    if (warp < kParts) {
      auto score2 = [&](const KV& r, int c0) {
#pragma unroll
        for (int u2 = 0; u2 < 2; ++u2) {
          const int seq = c0 + u2;
          if (seq < n) {
            float kf[16];
            up8<F16>(r.ka[u2], kf);
            up8<F16>(r.kb[u2], kf + 8);
            const float* qp = qs + seq * kDh + qd * 16;
            float a = 0.f;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const float4 q4 = *reinterpret_cast<const float4*>(qp + 4 * i);
              a = fmaf(q4.x, kf[4 * i], a); a = fmaf(q4.y, kf[4 * i + 1], a);
              a = fmaf(q4.z, kf[4 * i + 2], a); a = fmaf(q4.w, kf[4 * i + 3], a);
            }
            a += __shfl_xor_sync(0xffffffffu, a, 1);
            a += __shfl_xor_sync(0xffffffffu, a, 2);
            const float dot = valid ? a * 0.125f : -INFINITY;
            float m = dot;
            m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, 4));
            m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, 8));
            m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, 16));
            const float pj = valid ? __expf(dot - m) : 0.f;
            float l = pj;
            l += __shfl_xor_sync(0xffffffffu, l, 4);
            l += __shfl_xor_sync(0xffffffffu, l, 8);
            l += __shfl_xor_sync(0xffffffffu, l, 16);
            float oa = 0.f, ob = 0.f;
#pragma unroll
            for (int u = 0; u < 8; ++u) {
              const float pu = __shfl_sync(0xffffffffu, pj, 4 * u);
              const float2 f = up2<F16>(r.vr[u2][u]);
              oa = fmaf(pu, f.x, oa);
              ob = fmaf(pu, f.y, ob);
            }
            float* pt = parts + (seq * kParts + part) * kPartFloats;
            if (lane == 0) { pt[0] = m; pt[1] = l; }
            *reinterpret_cast<float2*>(pt + 2 + 2 * lane) = make_float2(oa, ob);
          }
        }
      };
      for (int c0 = 0; c0 < n; c0 += 4) {
        load2(bufB, c0 + 2);
        score2(bufA, c0);
        load2(bufA, c0 + 4);
        score2(bufB, c0 + 2);
      }
    }
    __syncthreads();
    {      // merge the 14 parts of sequence `warp` (flash-style rescale); padded sequences give zeros
      float2 o = make_float2(0.f, 0.f);
      if (warp < n) {
        float M = -INFINITY;
#pragma unroll
        for (int w = 0; w < kParts; ++w) M = fmaxf(M, parts[(warp * kParts + w) * kPartFloats]);
        float l = 0.f;
#pragma unroll
        for (int w = 0; w < kParts; ++w) {
          const float* pt = parts + (warp * kParts + w) * kPartFloats;
          const float sc_w = pt[1] > 0.f ? __expf(pt[0] - M) : 0.f;
          const float2 t = *reinterpret_cast<const float2*>(pt + 2 + 2 * lane);
          l = fmaf(pt[1], sc_w, l);
          o.x = fmaf(t.x, sc_w, o.x);
          o.y = fmaf(t.y, sc_w, o.y);
        }
        const float inv = 1.0f / l;
        o.x *= inv; o.y *= inv;
      }
      *reinterpret_cast<uint32_t*>(cs + warp * kCPitch + 2 * lane) = pk2<F16>(o.x, o.y);
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");     // Wco slice
    __syncthreads();
    r0_stamp(p.trace, 3);

    // ---- phase 3: partial out-projection of this head's K-slice: po[s][c] = sum_{k<64} Wco[c][64h+k] ctx_h[s][k];
    // warp w owns the 16-row output tiles w and w + 16
    {
#pragma unroll
      for (int mi = 0; mi < 2; ++mi) {
        const int mt = warp + 16 * mi;
        float acc[2][4];
#pragma unroll
        for (int nt = 0; nt < 2; ++nt)
#pragma unroll
          for (int jj = 0; jj < 4; ++jj) acc[nt][jj] = 0.f;
        const bf16* arow = wo + (16 * mt + (lane & 7) + ((lane >> 3) & 1) * 8) * kWoPitch + (lane >> 4) * 8;
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
          uint32_t a[4];
          ldmatrix_x4(a, arow + 16 * ks);
#pragma unroll
          for (int nt = 0; nt < 2; ++nt) {
            if (nt < ntiles) {
              const bf16* brow = cs + (8 * nt + gid) * kCPitch + 16 * ks + tig * 2;
              mma16816<F16>(acc[nt], a, *reinterpret_cast<const uint32_t*>(brow), *reinterpret_cast<const uint32_t*>(brow + 8));
            }
          }
        }
#pragma unroll
        for (int nt = 0; nt < 2; ++nt) {
          if (nt < ntiles) {
            float* o0 = po + (8 * nt + 2 * tig) * kPoPitch + 16 * mt + gid;
            o0[0] = acc[nt][0]; o0[kPoPitch] = acc[nt][1];
            o0[8] = acc[nt][2]; o0[kPoPitch + 8] = acc[nt][3];
          }
        }
      }
    }
    r0_stamp(p.trace, 4);
    cluster_barrier();     // every CTA's partial projection is complete and visible cluster-wide
    r0_stamp(p.trace, 5);

    // ---- phase 4: CTA h finishes the rows of the group's sequences s = h, h + 8: thread = output column.  The 8 partial
    // projections of the row come over DSMEM (fixed order), + residual + bias, then an ordinary block LayerNorm (two-pass,
    // fp32) - no statistics exchange between CTAs.  The cluster barrier that lets the peers reuse / retire their po
    // buffers is ARRIVED at as soon as the remote values are in registers and only WAITED for after the row is stored.
    {
      const int c = tid;                        // kThreads == kD
      float v[2] = {0.f, 0.f};
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int sq = h + kHeads * u;
        if (sq < n) {
#pragma unroll
          for (int r = 0; r < kHeads; ++r) v[u] += ld_remote_f(remote_addr(po + sq * kPoPitch + c, r));
        }
      }
      asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
      const float bo = __ldg(p.bo + c), gg = __ldg(p.g + c), bb = __ldg(p.be + c);
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int sq = h + kHeads * u;
        if (sq < n) {                             // uniform over the CTA
          const bf16 xh = xs[sq * kXPitch + c];
          float xr;
          if constexpr (F16) xr = __half2float(*reinterpret_cast<const __half*>(&xh));
          else xr = __bfloat162float(xh);
          const float val = v[u] + (xr + bo);
          const float ps = wsum(val);
          if (lane == 0) st[u * 32 + warp] = ps;
          __syncthreads();
          float mean = 0.f;
#pragma unroll
          for (int w = 0; w < kThreads / 32; ++w) mean += st[u * 32 + w];
          mean *= (1.0f / kD);
          const float dlt = val - mean;
          const float pq = wsum(dlt * dlt);
          if (lane == 0) st[u * 32 + 16 + warp] = pq;
          __syncthreads();
          float var = 0.f;
#pragma unroll
          for (int w = 0; w < kThreads / 32; ++w) var += st[u * 32 + 16 + w];
          const float rstd = rsqrtf(var * (1.0f / kD) + 1e-5f);
          const float outv = dlt * rstd * gg + bb;
          bf16* dst = p.x + (int64_t)(s0 + sq) * p.T * kD + c;
          if constexpr (F16) { const __half hv = __float2half_rn(outv); *dst = *reinterpret_cast<const bf16*>(&hv); }
          else *dst = __float2bfloat16_rn(outv);
        }
      }
      r0_stamp(p.trace, 6);
      // every peer has finished reading this CTA's po: the next group may overwrite it / the CTA may retire
      asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
    }
  }
}

}  // namespace

int row0_fused_launch(const bf16* x0c, const bf16* Wq, const float* bq, const bf16* kv, const bf16* Wo, const float* bo,
                      const float* g, const float* be, bf16* x, int S, int T, int Tk, int H, int d, int fp16, cudaStream_t st) {
  MSMD_REQUIRE(d == kD && H == kHeads && Tk >= 1 && Tk <= kParts * kPartKeys,
               "row0_fused: built for d_model 512, 8 heads x 64 and <= 112 memory tokens (got %d, %d, %d)", d, H, Tk);
  Row0Params p{x0c, Wq, bq, kv, Wo, bo, g, be, x, S, T, Tk, nullptr};
#ifdef MSMD_ROW0_TRACE
  static unsigned long long* tbuf = nullptr;
  if (!tbuf) MSMD_CHECK_CUDA(cudaMalloc(&tbuf, 8 * 8));
  p.trace = tbuf;
#endif
  auto kern = fp16 ? row0_fused_kernel<true> : row0_fused_kernel<false>;
  static bool attr = false;
  if (!attr) {
    MSMD_CHECK_CUDA(cudaFuncSetAttribute(row0_fused_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem));
    MSMD_CHECK_CUDA(cudaFuncSetAttribute(row0_fused_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem));
    attr = true;
  }
  // clusters that can be co-resident (a cluster of 8 lives inside one GPC): more would only queue behind them
  static int max_clusters = 0;
  if (max_clusters == 0) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(kNumSMs / kHeads * kHeads);
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = kSmem;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = kHeads; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    int nc = 0;
    if (cudaOccupancyMaxActiveClusters(&nc, row0_fused_kernel<false>, &cfg) != cudaSuccess || nc < 1) {
      (void)cudaGetLastError();
      nc = kNumSMs / kHeads;
    }
    max_clusters = nc < kNumSMs / kHeads ? nc : kNumSMs / kHeads;
  }
  const int ncl = S < max_clusters ? S : max_clusters;
  ProfileScope prof("row0_fused", st);
  kern<<<ncl * kHeads, kThreads, kSmem, st>>>(p);
  MSMD_CHECK_LAUNCH();
#ifdef MSMD_ROW0_TRACE
  {
    static int calls = 0;
    if (++calls == 40) {
      unsigned long long hst[8];
      MSMD_CHECK_CUDA(cudaStreamSynchronize(st));
      MSMD_CHECK_CUDA(cudaMemcpy(hst, tbuf, sizeof(hst), cudaMemcpyDeviceToHost));
      fprintf(stderr, "[row0 trace] S=%d clusters=%d cycles since start: staged+x %lld | q-proj %lld | attention %lld | out-proj %lld | "
              "cluster barrier %lld | reduce+LN %lld\n", S, ncl, (long long)(hst[1] - hst[0]), (long long)(hst[2] - hst[1]),
              (long long)(hst[3] - hst[2]), (long long)(hst[4] - hst[3]), (long long)(hst[5] - hst[4]), (long long)(hst[6] - hst[5]));
    }
  }
#endif
  return MSMD_OK;
}

}  // namespace msmd
