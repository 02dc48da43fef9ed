// FLAME decode, tensor-core path (impl 0): fp32-grade three-pass fp16 tcgen05 GEMM over K = NB + 36 with the
// linear blend skinning as its epilogue.  Replaces lbs.py:185 (blend_shapes einsum), :200-204 (pose correctives)
// and :210-221 (per-vertex transform blend + apply) in ONE kernel; the reference materialises ~10 GB of
// intermediates at B = 8192 (T [B,V,16] alone is 2.6 GB), this kernel writes only the vertices.
//
//   tile      = 256 frames x 126 columns on a CTA PAIR (cta_group::2; 42 whole vertices; the MMA is issued with
//               N = 128, the last two columns are junk and never stored).  Each CTA stages its own 128 frames of
//               A and HALF of the basis tile.  TWO neighbouring column tiles are computed together ("super-tile"):
//               every k-block of A feeds both, so the operand bytes per tile drop from 48 KB to 32 KB per k-block per
//               SM.  The kernel is bound by the L2 -> SM delivery of its operands (ncu: 3.05 GB in 423 us = the
//               7.2 TB/s every TMA-fed kernel of this library tops out at, tensor pipe 42% active), not by the MMAs.
//   operands  = two-term fp16 splits s x = hi + lo (22 mantissa bits; flame.cuh) of A [B,Kpad] (betas |
//               vec(R-I) | 0) and of the basis [3V,Kpad], K-major, TMA -> 128B-swizzled smem, 2 stages x 64 KB of
//               64-deep k-blocks.  (The tf32 hi/lo version of this kernel was bound by shared-memory bandwidth:
//               a K=8 tf32 MMA reads as many operand bytes as a K=16 fp16 one for half the FLOPs.)
//   MMA       = kind::f16 (fp16 in, fp32 accumulate), M256 N128 K16 issued by the leader CTA, three passes per
//               k-step and column tile: lo*hi, hi*lo, hi*hi into ONE accumulator (hi and lo carry the same scale).
//               Round 1 kept the cross terms in a second accumulator; sharing one costs ~3 more truncating
//               accumulations per k-step (measured error in tests/test_flame_gpu.py, bound 1e-5) and halves the
//               TMEM per tile, which is what lets two column tiles stay double-buffered.
//   TMEM      = per CTA 2 stages x 2 column tiles x 128 columns: the epilogue of super-tile i overlaps the MMAs of i+1
//   epilogue  = thread <-> frame: v_posed = acc / (sA sB) + template, T = sum_j w[v][j] * A_j[b] (5 joints x 12
//               coefficients held in registers), x = T [v_posed; 1]; staged through smem for coalesced stores
#include "flame.cuh"
#include "tc_common.cuh"
#include "profile.cuh"
#include <cstdlib>

namespace msmd {

namespace {

// k-block depth 64: 128-byte rows, SWIZZLE_128B, 2 stages x 64 KB.  The timeline shows the MMA loop waiting on operand
// delivery (20.5K cycles per super-tile for 10.8K cycles of MMA); 32-deep slots (64-byte rows, SWIZZLE_64B, 4 stages x
// 32 KB: the same 128 KB in flight) were tried to keep more fills in flight and measured SLOWER on the same box (350.6
// vs 337.8 us): the limit is the L2 -> SM delivery rate (~7.2 TB/s chip-wide), not slot granularity, and 64-byte rows
// double the request count.
constexpr int FT_BK = 64;
constexpr int FT_STAGES = 2, FT_NQ = 4, FT_G = 2;       // FT_G column tiles share every A k-block
constexpr int FT_BM = 128, FT_VERT = 42, FT_BN = 126, FT_UN = 128;
constexpr int FT_ROW_BYTES = FT_BK * 2;                  // one operand row of a k-block
constexpr int FT_TILE_BYTES = 128 * FT_ROW_BYTES;        // one operand tile: 128 rows
constexpr int FT_BHALF_BYTES = 64 * FT_ROW_BYTES;        // this CTA's half of a basis tile: 64 rows
__device__ __forceinline__ uint64_t ft_desc(uint32_t smem_addr) {
  return tc::make_smem_desc_sw128(smem_addr);
}
constexpr int FT_STAGE_BYTES = 2 * FT_TILE_BYTES + FT_G * 2 * FT_BHALF_BYTES;   // A_hi, A_lo, then per column tile: B_hi half, B_lo half
constexpr int FT_CHUNK_V = 8;                             // vertices per epilogue chunk (24 accumulator columns)
constexpr int FT_OUT_STRIDE = 127;                       // staging row stride (floats): odd -> conflict-free
constexpr int FT_EPI_WARPS = 8;                          // two warps per TMEM lane quarter, alternating chunks
constexpr int FT_EPI_Q_BYTES = 32 * FT_OUT_STRIDE * 4;    // one TMEM lane quarter (32 frames) x the tile's 126 columns
constexpr int FT_MISC_BYTES = 2048;                      // barriers, tmem slot
constexpr int FT_VC_FLOATS = (FT_VERT + 6) * 8;          // per-tile vertex constants (w0..w4 | template), padded to 48 vertices
constexpr int FT_SMEM_BYTES = 1024 + FT_STAGES * FT_STAGE_BYTES + FT_NQ * FT_EPI_Q_BYTES + FT_MISC_BYTES + 2 * FT_G * FT_VC_FLOATS * 4;
static_assert(FT_SMEM_BYTES <= 227 * 1024, "flame_tc shared memory");
constexpr int FT_THREADS = 64 + 32 * FT_EPI_WARPS;

struct FlameTcParams {
  CUtensorMap a_hi, a_lo, b_hi, b_lo;
  const float* vconst;   // [V(+pad), 8]  w0..w4 | template xyz
  const float* xf;       // [B,60]
  float* out;            // [B,3V]
  int B, V, N3, num_kb, tiles_m, tiles_n, tiles_n2;   // tiles_n2 = ceil(tiles_n / FT_G) super-tile columns
  unsigned long long* trace;   // -DMSMD_FLAME_TRACE builds: clock64 stamps of CTA 0, [role 0..2][tile 0..15][4]
};

__device__ __forceinline__ void ft_stamp(unsigned long long* tr, int role, int it, int ev) {
#ifdef MSMD_FLAME_TRACE
  if (tr != nullptr && blockIdx.x == 0 && it < 16) tr[(role * 16 + it) * 4 + ev] = clock64();
#endif
}

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* v) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}

__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t* v) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "r"(taddr)
               : "memory");
}

// NORM: every row of the skinning weights sums to 1, so T = A_0 + sum_{j>=1} w_j (A_j - A_0): 48 FMAs per vertex
// instead of 60 (the blend is the epilogue's - and the kernel's - critical path).
template <bool NORM>
__global__ void __launch_bounds__(FT_THREADS, 1) flame_tc_kernel(const __grid_constant__ FlameTcParams p) {
  using namespace tc;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* stage_base = smem;
  float* epi_base = reinterpret_cast<float*>(smem + FT_STAGES * FT_STAGE_BYTES);
  uint8_t* misc = reinterpret_cast<uint8_t*>(epi_base) + FT_NQ * FT_EPI_Q_BYTES;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(misc);  // [STAGES]
  uint64_t* empty_bar = full_bar + FT_STAGES;              // [STAGES]
  uint64_t* tfull_bar = empty_bar + FT_STAGES;             // [2]
  uint64_t* tempty_bar = tfull_bar + 2;                    // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);
  float* tile_w = reinterpret_cast<float*>(misc + FT_MISC_BYTES);  // [2][FT_G][48 vertices][8]: w0..w4 | template xyz
  constexpr int TILE_W_FLOATS = FT_VC_FLOATS;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int num_tiles = p.tiles_m * p.tiles_n2;     // super-tiles
  const int cta_rank = (int)cluster_ctarank();
  const int pair = (int)blockIdx.x / 2, npairs = (int)gridDim.x / 2;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&p.a_hi); prefetch_tmap(&p.a_lo); prefetch_tmap(&p.b_hi); prefetch_tmap(&p.b_lo);
    for (int s = 0; s < FT_STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(&tfull_bar[a], 1); mbar_init(&tempty_bar[a], 2 * FT_EPI_WARPS); }   // epilogue warps of both CTAs
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc_2sm(tmem_slot, 512);
  tc_fence_before();
  cluster_sync();   // the peer's barriers are initialised before anyone signals them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ---------------------------------------------------------------- TMA producer
    int s = 0, pit = 0;
    uint32_t ph = 0;
    for (int t = pair; t < num_tiles; t += npairs, ++pit) {
      const int m0 = (t / p.tiles_n2) * 2 * FT_BM + cta_rank * FT_BM, n0 = (t % p.tiles_n2) * FT_G * FT_BN + cta_rank * 64;
      for (int kb = 0; kb < p.num_kb; ++kb) {
        if (lane == 0) {
          if (kb == 0) ft_stamp(p.trace, 0, pit, 0);
          mbar_wait(&empty_bar[s], ph ^ 1);
          if (kb == 0) ft_stamp(p.trace, 0, pit, 1);
          if (kb == p.num_kb - 1) ft_stamp(p.trace, 0, pit, 2);
          uint8_t* st = stage_base + s * FT_STAGE_BYTES;
          // both CTAs' boxes land on the leader's barrier.  Rank 1's basis half covers tile columns 64..127: the
          // last two rows belong to the next tile (or are zero-filled past the end) and only feed junk columns.  A
          // column tile past the last one (odd tile count) reads zero rows / is zero-filled: its results are never stored.
          if (cta_rank == 0) mbar_expect_tx(&full_bar[s], 2 * FT_STAGE_BYTES);
          tma_load_2d_2sm(st, &p.a_hi, &full_bar[s], kb * FT_BK, m0);
          tma_load_2d_2sm(st + FT_TILE_BYTES, &p.a_lo, &full_bar[s], kb * FT_BK, m0);
#pragma unroll
          for (int g = 0; g < FT_G; ++g) {
            uint8_t* sb = st + 2 * FT_TILE_BYTES + g * 2 * FT_BHALF_BYTES;
            tma_load_2d_2sm(sb, &p.b_hi, &full_bar[s], kb * FT_BK, n0 + g * FT_BN);
            tma_load_2d_2sm(sb + FT_BHALF_BYTES, &p.b_lo, &full_bar[s], kb * FT_BK, n0 + g * FT_BN);
          }
        }
        __syncwarp();
        if (++s == FT_STAGES) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ---------------------------------------------------------------- MMA issuer
    constexpr uint32_t idesc = make_idesc(0, 2 * FT_BM, FT_UN);   // fp16 operands, fp32 accumulate
    int s = 0, it = 0;
    uint32_t ph = 0;
    for (int t = cta_rank == 0 ? pair : num_tiles; t < num_tiles; t += npairs, ++it) {   // leader only
      const int a = it & 1;
      const uint32_t aph = (it >> 1) & 1;
      const uint32_t d_acc = tmem_base + a * (FT_G * 128);
      if (lane == 0) {
        ft_stamp(p.trace, 1, it, 0);
        mbar_wait(&tempty_bar[a], aph ^ 1);
        tc_fence_after();
        ft_stamp(p.trace, 1, it, 1);
      }
      __syncwarp();
      for (int kb = 0; kb < p.num_kb; ++kb) {
        if (lane == 0) {
          mbar_wait(&full_bar[s], ph);
          tc_fence_after();
          if (kb == 0) ft_stamp(p.trace, 1, it, 2);
          const uint32_t sa = smem_u32(stage_base + s * FT_STAGE_BYTES);
          const uint64_t ah = ft_desc(sa), al = ft_desc(sa + FT_TILE_BYTES);
#pragma unroll
          for (int k = 0; k < FT_BK / 16; ++k) {
            const uint32_t acc = (kb | k) != 0;
#pragma unroll
            for (int g = 0; g < FT_G; ++g) {
              const uint32_t sb = sa + 2 * FT_TILE_BYTES + g * 2 * FT_BHALF_BYTES;
              const uint64_t bh = ft_desc(sb), bl = ft_desc(sb + FT_BHALF_BYTES);
              const uint32_t d = d_acc + g * 128;
              umma_2sm(d, desc_advance(al, k * 32), desc_advance(bh, k * 32), idesc, acc);   // lo * hi
              umma_2sm(d, desc_advance(ah, k * 32), desc_advance(bl, k * 32), idesc, 1u);    // hi * lo
              umma_2sm(d, desc_advance(ah, k * 32), desc_advance(bh, k * 32), idesc, 1u);    // hi * hi
            }
          }
          umma_commit_2sm(&empty_bar[s]);
        }
        __syncwarp();
        if (++s == FT_STAGES) { s = 0; ph ^= 1; }
      }
      if (lane == 0) { ft_stamp(p.trace, 1, it, 3); umma_commit_2sm(&tfull_bar[a]); }
      __syncwarp();
    }
  } else {
    // ---------------------------------------------------------------- epilogue: skinning
    const int q = warp & 3;                     // TMEM lane quarter this warp may access
    const int half = (warp - 2) >> 2;           // which of the quarter's two warps: chunks half, half+2, ...
    float* stage = epi_base + (q % FT_NQ) * (FT_EPI_Q_BYTES / 4);   // shared by the quarter's two warps
    const int etid = threadIdx.x - 64;
    constexpr int EPI_THREADS = 32 * FT_EPI_WARPS;
    constexpr int NCHUNK = (FT_VERT + FT_CHUNK_V - 1) / FT_CHUNK_V;
    int it = 0;
    for (int t = pair; t < num_tiles; t += npairs, ++it) {
      const int m0 = (t / p.tiles_n2) * 2 * FT_BM + cta_rank * FT_BM;
      const int nt0 = (t % p.tiles_n2) * FT_G;                    // first column tile of the super-tile
      const int ng = min(FT_G, p.tiles_n - nt0);                  // column tiles that exist
      const int a = it & 1;
      const uint32_t aph = (it >> 1) & 1;
      // per-tile vertex constants -> smem (double-buffered by super-tile parity); 16-byte copies
      float* tw_all = tile_w + a * (FT_G * TILE_W_FLOATS);
      for (int i = etid; i < ng * (FT_VC_FLOATS / 4); i += EPI_THREADS) {
        const int g = i / (FT_VC_FLOATS / 4), r = i - g * (FT_VC_FLOATS / 4);
        const int v0g = (nt0 + g) * FT_VERT;
        reinterpret_cast<float4*>(tw_all + g * TILE_W_FLOATS)[r] = __ldg(reinterpret_cast<const float4*>(p.vconst + (int64_t)v0g * 8) + r);
      }
      // this thread's frame: 5 joints x (3x3 | t); with normalised weights joints 1..4 are kept as differences to joint 0
      const int row = m0 + q * 32 + lane;
      float xf[60];
      {
        const float4* src = reinterpret_cast<const float4*>(p.xf + (int64_t)min(row, p.B - 1) * 60);
#pragma unroll
        for (int i = 0; i < 15; ++i) {
          const float4 f = __ldg(src + i);
          xf[4 * i] = f.x; xf[4 * i + 1] = f.y; xf[4 * i + 2] = f.z; xf[4 * i + 3] = f.w;
        }
        if constexpr (NORM) {
#pragma unroll
          for (int j = 1; j < 5; ++j)
#pragma unroll
            for (int e = 0; e < 12; ++e) xf[j * 12 + e] -= xf[e];
        }
      }
      asm volatile("bar.sync 1, %0;" ::"n"(EPI_THREADS) : "memory");
      if (warp == 2 && lane == 0) ft_stamp(p.trace, 2, it, 0);
      mbar_wait(&tfull_bar[a], aph);
      tc_fence_after();
      if (warp == 2 && lane == 0) ft_stamp(p.trace, 2, it, 1);
#pragma unroll 1
      for (int g = 0; g < FT_G; ++g) {
        const float* tw = tw_all + g * TILE_W_FLOATS;
        const int n0 = (nt0 + g) * FT_BN;
        const uint32_t t_main = tmem_base + ((uint32_t)(q * 32) << 16) + a * (FT_G * 128) + g * 128;
        if (g < ng) {
          // 8-vertex chunks (24 accumulator columns); the last one (ck = 5) holds 2 vertices.  This warp takes chunks
          // half, half + 2, half + 4; the TMEM reads of its next chunk are in flight while the current one is skinned.
          auto load_chunk = [&](int ck, uint32_t (&m)[24]) {
            const int c0 = ck * 3 * FT_CHUNK_V;
            if (ck < NCHUNK - 1) {
              tmem_ld16(t_main + c0, m); tmem_ld8(t_main + c0 + 16, m + 16);
            } else {   // columns 120..125; an x16 load would run past the 128-column accumulator
              tmem_ld8(t_main + c0, m);
            }
          };
          auto skin_chunk = [&](int ck, const uint32_t (&m)[24]) {
            const int nv = min(FT_CHUNK_V, FT_VERT - ck * FT_CHUNK_V);
#pragma unroll
            for (int v = 0; v < FT_CHUNK_V; ++v) {
              if (v < nv) {
                const int vv = ck * FT_CHUNK_V + v, cc = 3 * vv;
                const float4 wa = *reinterpret_cast<const float4*>(tw + vv * 8);       // w0 w1 w2 w3   (broadcast)
                const float4 wb = *reinterpret_cast<const float4*>(tw + vv * 8 + 4);   // w4 tx ty tz
                constexpr float kInv = 1.0f / (kFlameScaleA * kFlameScaleB);            // the operands carried these scales
                const float px = fmaf(__uint_as_float(m[3 * v]), kInv, wb.y);
                const float py = fmaf(__uint_as_float(m[3 * v + 1]), kInv, wb.z);
                const float pz = fmaf(__uint_as_float(m[3 * v + 2]), kInv, wb.w);
                float T[12];
#pragma unroll
                for (int e = 0; e < 12; ++e) {
                  float s = NORM ? xf[e] : wa.x * xf[e];
                  s = fmaf(wa.y, xf[12 + e], s);
                  s = fmaf(wa.z, xf[24 + e], s);
                  s = fmaf(wa.w, xf[36 + e], s);
                  T[e] = fmaf(wb.x, xf[48 + e], s);
                }
                stage[lane * FT_OUT_STRIDE + cc + 0] = fmaf(T[0], px, fmaf(T[1], py, fmaf(T[2], pz, T[9])));
                stage[lane * FT_OUT_STRIDE + cc + 1] = fmaf(T[3], px, fmaf(T[4], py, fmaf(T[5], pz, T[10])));
                stage[lane * FT_OUT_STRIDE + cc + 2] = fmaf(T[6], px, fmaf(T[7], py, fmaf(T[8], pz, T[11])));
              }
            }
          };
          {
            uint32_t mA[24], mB[24];
            load_chunk(half, mA);
            tmem_ld_wait();
            load_chunk(half + 2, mB);
            skin_chunk(half, mA);
            tmem_ld_wait();
            load_chunk(half + 4, mA);
            skin_chunk(half + 2, mB);
            tmem_ld_wait();
            skin_chunk(half + 4, mA);
          }
        }
        if (g == FT_G - 1) {
          if (warp == 2 && lane == 0) ft_stamp(p.trace, 2, it, 2);
          tc_fence_before();
          __syncwarp();
          if (lane == 0) {   // accumulators are consumed: the MMAs of the next super-tile may overwrite them during the stores
            if (cta_rank != 0) mbar_arrive_cluster(&tempty_bar[a], 0);   // the leader's MMA warp waits for both CTAs
            else mbar_arrive(&tempty_bar[a]);
          }
        }
        // both warps of the quarter have staged their vertices: store whole 504-byte tile rows, coalesced; four rows'
        // shared-memory reads are issued together so the stores stream instead of paying one LDS latency per row
        asm volatile("bar.sync %0, 64;" ::"r"(2 + q) : "memory");
        if (g < ng) {
          const int ncol = min(FT_BN, p.N3 - n0);
#pragma unroll 1
          for (int r0 = half; r0 < 32; r0 += 8) {
            float val[4][4];
#pragma unroll
            for (int u = 0; u < 4; ++u)
#pragma unroll
              for (int k = 0; k < 4; ++k) val[u][k] = (lane + 32 * k < FT_BN) ? stage[(r0 + 2 * u) * FT_OUT_STRIDE + lane + 32 * k] : 0.f;
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const int grow = m0 + q * 32 + r0 + 2 * u;
              if (grow < p.B) {
                float* dst = p.out + (int64_t)grow * p.N3 + n0;
#pragma unroll
                for (int k = 0; k < 4; ++k)
                  if (lane + 32 * k < ncol) __stcs(dst + lane + 32 * k, val[u][k]);
              }
            }
          }
        }
        // the quarter's staging buffer is rewritten by the next column tile: both warps are done reading it
        asm volatile("bar.sync %0, 64;" ::"r"(2 + q) : "memory");
      }
      if (warp == 2 && lane == 0) ft_stamp(p.trace, 2, it, 3);
    }
  }

  tc_fence_before();
  cluster_sync();   // the peer may still be reading this CTA's smem / signalling its barriers
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_2sm(tmem_base, 512);
  }
}

}  // namespace

int flame_decode_tc(msmd_flame* fh, int64_t B, float* verts_out, cudaStream_t st) {
  FlameTcParams p;
  memset(&p, 0, sizeof(p));
  const int64_t rows = fh->cap_B;  // workspace rows (multiple of 128)
  int rc;
  const auto f32 = CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
  const uint64_t ldk = (uint64_t)fh->Kpad * 2;
  const auto FT_SWZ = CU_TENSOR_MAP_SWIZZLE_128B;
  if ((rc = make_tmap_2d(&p.a_hi, fh->A_hi, f32, fh->Kpad, rows, ldk, FT_BK, FT_BM, FT_SWZ))) return rc;
  if ((rc = make_tmap_2d(&p.a_lo, fh->A_lo, f32, fh->Kpad, rows, ldk, FT_BK, FT_BM, FT_SWZ))) return rc;
  if ((rc = make_tmap_2d(&p.b_hi, fh->basis_hi, f32, fh->Kpad, fh->N3pad, ldk, FT_BK, 64, FT_SWZ))) return rc;
  if ((rc = make_tmap_2d(&p.b_lo, fh->basis_lo, f32, fh->Kpad, fh->N3pad, ldk, FT_BK, 64, FT_SWZ))) return rc;
  p.vconst = fh->vconst; p.xf = fh->xf; p.out = verts_out;
  p.B = (int)B; p.V = fh->V; p.N3 = fh->N3; p.num_kb = fh->Kpad / FT_BK;
  p.tiles_m = cdiv(B, 2 * FT_BM);
  p.tiles_n = cdiv(fh->N3, FT_BN);
  p.tiles_n2 = cdiv(p.tiles_n, FT_G);
  static bool attr = false;
  if (!attr) {
    MSMD_CHECK_CUDA(cudaFuncSetAttribute(flame_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, FT_SMEM_BYTES));
    MSMD_CHECK_CUDA(cudaFuncSetAttribute(flame_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, FT_SMEM_BYTES));
    attr = true;
  }
  const int tiles = p.tiles_m * p.tiles_n2;
  ProfileScope prof("flame_fused", st);
  const int pairs = tiles < kNumSMs / 2 ? tiles : kNumSMs / 2;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2 * pairs);
  cfg.blockDim = dim3(FT_THREADS);
  cfg.dynamicSmemBytes = FT_SMEM_BYTES;
  cfg.stream = st;
  cudaLaunchAttribute attr_c[1];
  attr_c[0].id = cudaLaunchAttributeClusterDimension;
  attr_c[0].val.clusterDim.x = 2; attr_c[0].val.clusterDim.y = 1; attr_c[0].val.clusterDim.z = 1;
  cfg.attrs = attr_c;
  cfg.numAttrs = 1;
#ifdef MSMD_FLAME_TRACE
  static unsigned long long* tbuf = nullptr;
  if (!tbuf) MSMD_CHECK_CUDA(cudaMalloc(&tbuf, 3 * 16 * 4 * 8));
  MSMD_CHECK_CUDA(cudaMemsetAsync(tbuf, 0, 3 * 16 * 4 * 8, st));
  p.trace = tbuf;
#endif
  if (fh->weights_normalised) MSMD_CHECK_CUDA(cudaLaunchKernelEx(&cfg, flame_tc_kernel<true>, p));
  else MSMD_CHECK_CUDA(cudaLaunchKernelEx(&cfg, flame_tc_kernel<false>, p));
  MSMD_CHECK_LAUNCH();
#ifdef MSMD_FLAME_TRACE
  {
    static int calls = 0;
    if (++calls == 10) {
      unsigned long long h[3 * 16 * 4];
      MSMD_CHECK_CUDA(cudaStreamSynchronize(st));
      MSMD_CHECK_CUDA(cudaMemcpy(h, tbuf, sizeof(h), cudaMemcpyDeviceToHost));
      const unsigned long long t0 = h[0];
      const char* names[3] = {"tma  [tile start, slot free, last kb issued]", "mma  [start, acc free, first full, last issued]",
                              "epi  [start, acc full, computed, stored]"};
      for (int r = 0; r < 3; ++r) {
        fprintf(stderr, "[flame trace] %s\n", names[r]);
        for (int j = 0; j < 10; ++j) {
          const unsigned long long* e = &h[(r * 16 + j) * 4];
          fprintf(stderr, "   tile %2d: %7lld %7lld %7lld %7lld\n", j, (long long)(e[0] - t0), (long long)(e[1] - t0),
                  (long long)(e[2] ? e[2] - t0 : 0), (long long)(e[3] ? e[3] - t0 : 0));
        }
      }
    }
  }
#endif
  return MSMD_OK;
}

void flame_tc_destroy(msmd_flame* fh) { (void)fh; }

}  // namespace msmd
