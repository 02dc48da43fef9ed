// Self-attention of the decoder layers on tcgen05 (nn.TransformerDecoderLayer._sa_block -> nn.MultiheadAttention,
// no mask: DenoisingNetwork_MSMD.forward passes tgt_mask=None, model.py:951-958), and, as the CROSS instantiation, the
// banded cross-attention (_mha_block with memory_mask = alignment_mask, model.py:879-883) that every align_mask_width
// other than 1 needs on every step: Q from its own [S*T, d] buffer, K|V from the per-window cache [S*Tk, 2d].
//
// One "job" = one (sequence, head): S = Q K^T (128 x 112 x 64), row softmax, O = P V (128 x 64 x 112), T <= 112
// tokens so a sequence is a single tile and there is no online-softmax rescaling.  The legacy mma.sync path
// runs at 1/16 of the tcgen05 rate on this chip and bound the previous kernel (HMMA sub-pipe 87% busy, 33 us per
// layer); here the two GEMMs cost ~450 tensor cycles per job and the kernel is bound by HBM (q,k,v in, ctx out)
// and by the softmax's MUFU.EX2.
//
// Persistent CTA per SM, 10 warps:
//   warp 0      TMA producer: Q [128 x 64], K [112 x 64], V [112 x 64] boxes of the packed qkv rows -> 3-stage ring
//   warp 1      MMA issuer:  S_g = Q K^T  (K-major A and B), then O_g = P_g V with V as an MN-major B operand
//               (the [key][dh] rows TMA wrote ARE the MN-major SWIZZLE_128B canonical layout: 8-key groups 1024 B apart)
//   warps 2-5   softmax group 0 (even jobs), warps 6-9 softmax group 1 (odd jobs): thread = query row;
//               TMEM -> registers, exp2, P (bf16) -> swizzled shared memory as the K-major A operand of P V,
//               later O / rowsum -> the (free again) P buffer -> one TMA store of the [T x 64] head slice.
//               The two groups ping-pong so one computes while the other waits on its MMA.
// A CTA owns a contiguous range of jobs (consecutive heads of the same sequences: the 128-byte head slices of one
// qkv row are fetched close together in time).
// TMEM: per group S at columns [0,112) and O at [128,192) of a 192-column slice.
#include "denoiser_kernels.cuh"
#include "profile.cuh"
#include "tc_common.cuh"
#include <cstdlib>

namespace msmd {
namespace {

using namespace tc;

constexpr int kKeys = 112;                       // key tile: N of Q K^T, K of P V
constexpr int kStages = 3;
constexpr int kQBytes = 128 * 128, kKVBytes = kKeys * 128;
constexpr int kStageBytes = kQBytes + 2 * kKVBytes;          // 45056
constexpr int kPBytes = 2 * 128 * 128;                       // two 64-key column blocks of [128 rows][128 B]
constexpr int kBarBytes = 256;
constexpr int kSmemBytes = 1024 + kStages * kStageBytes + 2 * kPBytes + kBarBytes;
constexpr int kThreads = 320;
constexpr int kGroupCols = 192;                  // TMEM columns per softmax group (S: 128, O: 64)

struct AttnParams {
  CUtensorMap q_map, kv_map;
  CUtensorMap out_map;     // ctx rows, box {64 head dims, T rows}: a job's store covers exactly its sequence
  int S, T, H, jobs;
  unsigned long long* trace;   // -DMSMD_ATTN_TRACE builds: clock64 stamps of CTA 0, [role 0..2][job 0..15][8]
  int Tk, width;               // CROSS: keys per sequence, alignment band (0 = no band)
};

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* v) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}

__device__ __forceinline__ float ex2(float x) {      // one MUFU.EX2 (exp2f wraps it in a denormal-range fix-up: 3 more instructions)
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
template <bool F16>
__device__ __forceinline__ uint32_t pack16(float a, float b) {
  if constexpr (F16) {
    __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
  } else {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
  }
}

__device__ __forceinline__ void attn_stamp(unsigned long long* tr, int role, int job, int ev) {
#ifdef MSMD_ATTN_TRACE
  if (tr != nullptr && blockIdx.x == 0 && job < 16) tr[(role * 16 + job) * 8 + ev] = clock64();
#endif
}

// CROSS = false: q|k|v rows of one packed [S*T, 3d] buffer, every key visible (keys >= T masked; TAIL16: T > kKeys - 16).
// CROSS = true: q [S*T, d], k|v [S*Tk, 2d]; token 0 sees every key, token r >= 1 sees key c iff |c - (r-1)| <= width-1
// (width 0: every key).  The 112-key tile covers Tk <= 112 keys; the rows past Tk (next sequence / TMA zero fill) are
// masked.  TAIL16 is unused.
template <bool TAIL16, bool F16, bool CROSS>
__global__ void __launch_bounds__(kThreads, 1) self_attn_tc_kernel(const __grid_constant__ AttnParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* stage_base = smem;
  uint8_t* p_base = smem + kStages * kStageBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(p_base + 2 * kPBytes);
  uint64_t* full_bar = bars;                  // [kStages]
  uint64_t* empty_bar = bars + kStages;       // [kStages]
  uint64_t* sfull_bar = bars + 2 * kStages;   // [2]  S_g complete in TMEM
  uint64_t* pfull_bar = sfull_bar + 2;        // [2]  P_g written to shared memory
  uint64_t* ofull_bar = pfull_bar + 2;        // [2]  O_g complete in TMEM
  uint64_t* aempty_bar = ofull_bar + 2;       // [2]  S_g / O_g read out: the group's TMEM slice may be overwritten
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(aempty_bar + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int d = p.H * 64;
  // contiguous job range of this CTA
  const int job0 = (int)(((int64_t)p.jobs * blockIdx.x) / gridDim.x);
  const int njobs = (int)(((int64_t)p.jobs * (blockIdx.x + 1)) / gridDim.x) - job0;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&p.q_map);
    prefetch_tmap(&p.kv_map);
    prefetch_tmap(&p.out_map);
    for (int s = 0; s < kStages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    for (int g = 0; g < 2; ++g) {
      mbar_init(&sfull_bar[g], 1); mbar_init(&pfull_bar[g], 4); mbar_init(&ofull_bar[g], 1); mbar_init(&aempty_bar[g], 4);
    }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    if (lane == 0) {
      for (int i = 0; i < njobs; ++i) {
        const int job = job0 + i;
        const int s = job / p.H, h = job % p.H;
        const int st = i % kStages;
        mbar_wait(&empty_bar[st], ((i / kStages) & 1) ^ 1);
        uint8_t* sq = stage_base + st * kStageBytes;
        mbar_expect_tx(&full_bar[st], kStageBytes);
        tma_load_2d(sq, &p.q_map, &full_bar[st], h * 64, s * p.T);
        if constexpr (CROSS) {
          tma_load_2d(sq + kQBytes, &p.kv_map, &full_bar[st], h * 64, s * p.Tk);
          tma_load_2d(sq + kQBytes + kKVBytes, &p.kv_map, &full_bar[st], d + h * 64, s * p.Tk);
        } else {
          tma_load_2d(sq + kQBytes, &p.kv_map, &full_bar[st], d + h * 64, s * p.T);
          tma_load_2d(sq + kQBytes + kKVBytes, &p.kv_map, &full_bar[st], 2 * d + h * 64, s * p.T);
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    constexpr uint32_t idesc_qk = make_idesc(F16 ? 0 : 1, 128, kKeys);                 // bf16 / fp16, K-major A and B
    constexpr uint32_t idesc_pv = make_idesc(F16 ? 0 : 1, 128, 64) | (1u << 16);       // B (= V) is MN-major
    if (lane == 0) {
      for (int i = 0; i <= njobs; ++i) {
        if (i < njobs) {   // S_g = Q K^T of job i
          const int st = i % kStages, g = i & 1;
          mbar_wait(&full_bar[st], (i / kStages) & 1);
          mbar_wait(&aempty_bar[g], ((i >> 1) & 1) ^ 1);
          tc_fence_after();
          const uint32_t sq = smem_u32(stage_base + st * kStageBytes);
          const uint64_t dq = make_smem_desc_sw128(sq), dk = make_smem_desc_sw128(sq + kQBytes);
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma<0>(tmem_base + g * kGroupCols, desc_advance(dq, k * 32), desc_advance(dk, k * 32), idesc_qk, k != 0);
          umma_commit(&sfull_bar[g]);
          attn_stamp(p.trace, 0, i, 0);
        }
        if (i >= 1) {      // O_g = P_g V of job i-1
          const int j = i - 1, st = j % kStages, g = j & 1;
          attn_stamp(p.trace, 0, j, 1);
          mbar_wait(&pfull_bar[g], (j >> 1) & 1);
          tc_fence_after();
          attn_stamp(p.trace, 0, j, 2);
          const uint32_t sv = smem_u32(stage_base + st * kStageBytes + kQBytes + kKVBytes);
          const uint32_t sp = smem_u32(p_base + g * kPBytes);
#pragma unroll
          for (int ks = 0; ks < kKeys / 16; ++ks) {
            const uint64_t dp = make_smem_desc_sw128(sp + (ks >> 2) * (128 * 128) + (ks & 3) * 32);
            const uint64_t dv = make_smem_desc_sw128(sv + ks * 2048);       // 16 keys = two 8-key groups of 1024 B
            umma<0>(tmem_base + g * kGroupCols + 128, dp, dv, idesc_pv, ks != 0);
          }
          umma_commit(&ofull_bar[g]);
          umma_commit(&empty_bar[st]);   // Q, K (read by the earlier MMAs) and V of this stage are free
          attn_stamp(p.trace, 0, j, 3);
        }
      }
    }
    __syncwarp();
  } else {
    // ------------------------------------------------------------------ softmax + output (thread = query row)
    const int g = (warp - 2) >> 2;
    const int q = warp & 3;                       // TMEM lane quarter this warp may access
    const int r = q * 32 + lane;                  // query row of the tile
    const uint32_t t_s = tmem_base + ((uint32_t)(q * 32) << 16) + g * kGroupCols;
    const uint32_t t_o = t_s + 128;
    uint8_t* prow = p_base + g * kPBytes + r * 128;
    const int swz = r & 7;
    const float kScale = 0.125f * 1.4426950408889634f;   // 1/sqrt(64) * log2(e)
    const bool issuer = (warp - 2) % 4 == 0 && lane == 0;   // one thread per group owns the group's TMA stores
    // CROSS: visible keys of this row as a bit mask over the 112-key tile (bit c of vis[c / 32]).  Token 0, the no-band
    // case and the tile rows past T (never stored) see all Tk keys; a motion row always sees its own column r-1 < Tk.
    uint32_t vis[(kKeys + 31) / 32] = {};
    if constexpr (CROSS) {
      int lo = 0, hi = p.Tk - 1;
      if (p.width > 0 && r >= 1 && r < p.T) { lo = max(0, r - p.width); hi = min(hi, r + p.width - 2); }
#pragma unroll
      for (int k = 0; k < (kKeys + 31) / 32; ++k) {
        const int a = max(lo - 32 * k, 0), b = min(hi - 32 * k, 31);
        vis[k] = a <= b ? (0xffffffffu >> (31 - b + a)) << a : 0u;
      }
    }
    for (int i = g, it = 0; i < njobs; i += 2, ++it) {
      const int job = job0 + i;
      const int s = job / p.H, h = job % p.H;
      const uint32_t ph = it & 1;
      const bool tr0 = issuer;
      if (tr0) attn_stamp(p.trace, 1 + g, i, 0);
      mbar_wait(&sfull_bar[g], ph);
      tc_fence_after();
      if (tr0) attn_stamp(p.trace, 1 + g, i, 1);
      uint32_t v[kKeys];
      tmem_ld32(t_s, v);
      tmem_ld32(t_s + 32, v + 32);
      tmem_ld32(t_s + 64, v + 64);
      tmem_ld16(t_s + 96, v + 96);
      tmem_ld_wait();
      if (tr0) attn_stamp(p.trace, 1 + g, i, 2);
      float m = -INFINITY;
#pragma unroll
      for (int c = 0; c < kKeys; ++c) {
        if constexpr (CROSS) {
          const float x = (vis[c >> 5] >> (c & 31)) & 1u ? __uint_as_float(v[c]) : -INFINITY;
          v[c] = __float_as_uint(x);
        } else if (c >= kKeys - 16 || !TAIL16) {   // only the last 16 key columns can lie beyond T (TAIL16: T > kKeys - 16)
          const float x = c < p.T ? __uint_as_float(v[c]) : -INFINITY;
          v[c] = __float_as_uint(x);
        }
        m = fmaxf(m, __uint_as_float(v[c]));
      }
      const float ms = m * kScale;
      // the previous job's output store has finished reading this group's P buffer
      if (issuer) tma_store_wait_read<0>();
      asm volatile("bar.sync %0, 128;" ::"r"(1 + g) : "memory");
      float l = 0.f;
#pragma unroll
      for (int kc = 0; kc < kKeys / 8; ++kc) {
        uint32_t w[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const float e0 = ex2(fmaf(__uint_as_float(v[kc * 8 + 2 * u]), kScale, -ms));
          const float e1 = ex2(fmaf(__uint_as_float(v[kc * 8 + 2 * u + 1]), kScale, -ms));
          l += e0 + e1;
          w[u] = pack16<F16>(e0, e1);
        }
        *reinterpret_cast<uint4*>(prow + (kc >> 3) * (128 * 128) + (((kc & 7) ^ swz) << 4)) = make_uint4(w[0], w[1], w[2], w[3]);
      }
      fence_proxy_async_smem();     // P (generic-proxy writes) -> visible to the MMA's async-proxy reads
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&pfull_bar[g]);
      if (tr0) attn_stamp(p.trace, 1 + g, i, 3);

      mbar_wait(&ofull_bar[g], ph);   // P V done: O_g is complete and P_g is no longer read
      tc_fence_after();
      if (tr0) attn_stamp(p.trace, 1 + g, i, 4);
      uint32_t o[64];
      tmem_ld32(t_o, o);
      tmem_ld32(t_o + 32, o + 32);
      tmem_ld_wait();
      tc_fence_before();   // S_g and O_g are both in registers: hand the group's TMEM slice back (releasing S_g earlier,
      __syncwarp();        // right after its read, was measured: no change)
      if (lane == 0) mbar_arrive(&aempty_bar[g]);
      const float inv = 1.0f / l;
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        uint32_t w[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          w[u] = pack16<F16>(__uint_as_float(o[c * 8 + 2 * u]) * inv, __uint_as_float(o[c * 8 + 2 * u + 1]) * inv);
        }
        *reinterpret_cast<uint4*>(prow + ((c ^ swz) << 4)) = make_uint4(w[0], w[1], w[2], w[3]);   // first 64-key block of P_g
      }
      fence_proxy_async_smem();
      asm volatile("bar.sync %0, 128;" ::"r"(1 + g) : "memory");
      if (issuer) {
        tma_store_2d(&p.out_map, p_base + g * kPBytes, h * 64, s * p.T);
        tma_store_commit();
        attn_stamp(p.trace, 1 + g, i, 5);
      }
    }
    if (issuer) tma_store_wait<0>();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

}  // namespace

int self_attn_tc_launch(const bf16* qkv, bf16* ctx, int S, int T, int H, int fp16, cudaStream_t st) {
  MSMD_REQUIRE(T >= 1 && T <= kKeys, "self_attn: sequence length %d exceeds the %d-token tile", T, kKeys);
  MSMD_REQUIRE(H >= 1 && S >= 1, "self_attn: empty problem");
  AttnParams p;
  memset(&p, 0, sizeof(p));
  const int d = H * 64;
  int rc;
  const auto dt16 = fp16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  const uint64_t rows = (uint64_t)S * T;
  if ((rc = make_tmap_2d(&p.q_map, qkv, dt16, 3 * d, rows, (uint64_t)3 * d * 2, 64, 128,
                         CU_TENSOR_MAP_SWIZZLE_128B)))
    return rc;
  if ((rc = make_tmap_2d(&p.kv_map, qkv, dt16, 3 * d, rows, (uint64_t)3 * d * 2, 64, kKeys,
                         CU_TENSOR_MAP_SWIZZLE_128B)))
    return rc;
  if ((rc = make_tmap_2d(&p.out_map, ctx, dt16, d, rows, (uint64_t)d * 2, 64, T,
                         CU_TENSOR_MAP_SWIZZLE_128B)))
    return rc;
  p.S = S; p.T = T; p.H = H; p.jobs = S * H;
#ifdef MSMD_ATTN_TRACE
  static unsigned long long* tbuf = nullptr;
  if (!tbuf) MSMD_CHECK_CUDA(cudaMalloc(&tbuf, 3 * 16 * 8 * 8));
  MSMD_CHECK_CUDA(cudaMemsetAsync(tbuf, 0, 3 * 16 * 8 * 8, st));
  p.trace = tbuf;
#endif
  static bool attr = false;
  if (!attr) {
    MSMD_CHECK_CUDA(cudaFuncSetAttribute(self_attn_tc_kernel<true, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
    MSMD_CHECK_CUDA(cudaFuncSetAttribute(self_attn_tc_kernel<false, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
    MSMD_CHECK_CUDA(cudaFuncSetAttribute(self_attn_tc_kernel<true, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
    MSMD_CHECK_CUDA(cudaFuncSetAttribute(self_attn_tc_kernel<false, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
    attr = true;
  }
  ProfileScope prof("self_attn", st);
  const int grid = p.jobs < kNumSMs ? p.jobs : kNumSMs;
  auto kern = T > kKeys - 16 ? (fp16 ? self_attn_tc_kernel<true, true, false> : self_attn_tc_kernel<true, false, false>)
                             : (fp16 ? self_attn_tc_kernel<false, true, false> : self_attn_tc_kernel<false, false, false>);
  kern<<<grid, kThreads, kSmemBytes, st>>>(p);
  MSMD_CHECK_LAUNCH();
#ifdef MSMD_ATTN_TRACE
  {
    static int dumps = 0;
    unsigned long long h[3 * 16 * 8];
    MSMD_CHECK_CUDA(cudaStreamSynchronize(st));
    MSMD_CHECK_CUDA(cudaMemcpy(h, tbuf, sizeof(h), cudaMemcpyDeviceToHost));
    if (dumps++ == 20) {
      const unsigned long long t0 = h[0];
      const char* names[3] = {"mma   [QK issued, wait P, got P, PV issued]", "grp0  [wait S, got S, S in regs, P arrived, got O, store issued]",
                              "grp1  [same]"};
      for (int r = 0; r < 3; ++r) {
        fprintf(stderr, "[attn trace] %s\n", names[r]);
        for (int j = 0; j < 12; ++j) {
          const unsigned long long* e = &h[(r * 16 + j) * 8];
          if (!e[0] && !e[1] && !e[2]) continue;
          fprintf(stderr, "   job %2d:", j);
          for (int k = 0; k < 6; ++k) fprintf(stderr, " %7lld", e[k] ? (long long)(e[k] - t0) : -1LL);
          fprintf(stderr, "\n");
        }
      }
    }
  }
#endif
  return MSMD_OK;
}

int cross_attn_tc_launch(const bf16* q, const bf16* kv, bf16* ctx, int S, int T, int Tk, int H, int width, int fp16,
                         cudaStream_t st) {
  MSMD_REQUIRE(T >= 2 && T <= kKeys && Tk >= T - 1 && Tk <= kKeys,
               "cross_attn: %d queries / %d keys exceed the %d-token tile (or a motion row has no key)", T, Tk, kKeys);
  MSMD_REQUIRE(H >= 1 && S >= 1 && width >= 0, "cross_attn: empty problem or negative band width");
  AttnParams p;
  memset(&p, 0, sizeof(p));
  const int d = H * 64;
  int rc;
  const auto dt16 = fp16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  const uint64_t rows = (uint64_t)S * T, krows = (uint64_t)S * Tk;
  if ((rc = make_tmap_2d(&p.q_map, q, dt16, d, rows, (uint64_t)d * 2, 64, 128, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  if ((rc = make_tmap_2d(&p.kv_map, kv, dt16, 2 * d, krows, (uint64_t)2 * d * 2, 64, kKeys, CU_TENSOR_MAP_SWIZZLE_128B)))
    return rc;
  if ((rc = make_tmap_2d(&p.out_map, ctx, dt16, d, rows, (uint64_t)d * 2, 64, T, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  p.S = S; p.T = T; p.H = H; p.jobs = S * H; p.Tk = Tk; p.width = width;
  static bool attr = false;
  if (!attr) {
    MSMD_CHECK_CUDA(cudaFuncSetAttribute(self_attn_tc_kernel<true, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
    MSMD_CHECK_CUDA(cudaFuncSetAttribute(self_attn_tc_kernel<true, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
    attr = true;
  }
  ProfileScope prof("cross_attn", st);
  const int grid = p.jobs < kNumSMs ? p.jobs : kNumSMs;
  auto kern = fp16 ? self_attn_tc_kernel<true, true, true> : self_attn_tc_kernel<true, false, true>;
  kern<<<grid, kThreads, kSmemBytes, st>>>(p);
  MSMD_CHECK_LAUNCH();
  return MSMD_OK;
}

}  // namespace msmd
