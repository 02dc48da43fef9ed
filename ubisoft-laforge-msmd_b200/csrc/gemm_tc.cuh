// tcgen05 / TMEM / TMA GEMM core:  out[M,N] = act(A[M,K] . W[N,K]^T + bias) (+ aux)
//
// Both operands are K-major (nn.Linear layout), fetched by TMA into 128-byte-swizzled shared-memory
// tiles and multiplied by tcgen05.mma with the fp32 accumulator in TMEM.  Warp roles (one CTA per SM,
// persistent over tiles):   warp 0 = TMA producer, warp 1 = MMA issuer + TMEM owner,
// warps 2.. = epilogue (TMEM -> registers -> swizzled smem -> TMA store), double-buffered accumulators
// so the epilogue of tile i overlaps the MMAs of tile i+1.
//
// MODE 0: bf16 operands, one pass (kind::f16).
// MODE 1: fp32-grade "tf32x3": operands pre-split into hi (tf32-exact) + lo (remainder); three
//         kind::tf32 MMAs per k-step (hi*hi + hi*lo + lo*hi), error ~2^-21 relative.
// MODE 2: fp32-grade "fp16x3": operands pre-split into fp16 hi + fp16 lo with x = hi + 2^-11 lo (22 mantissa bits,
//         msmd_split_f16); three kind::f16 MMAs per k-step, the cross terms rescaled in the epilogue.  Half the MMA
//         instructions and operand bytes of MODE 1 (a K=8 tf32 MMA moves as many bytes as a K=16 fp16 one), but
//         |x| must stay below the fp16 range (65504).
// MODE 3: fp16 operands, one pass (kind::f16, fp16 in / fp16 out): the tensor-core cost of MODE 0 with 11 mantissa
//         bits instead of 8 - the sampler's intermediate-precision steps (x0_hat error 8e-4 instead of 6.5e-3).
#pragma once
#include "common.cuh"
#include "tc_common.cuh"
#include <cuda_bf16.h>
#include <cuda_fp16.h>

namespace msmd {

struct GemmParams {
  CUtensorMap a_map, b_map;        // MODE 0: bf16 A / W.  MODE 1: hi parts (fp32)
  CUtensorMap a_lo_map, b_lo_map;  // MODE 1 only
  CUtensorMap out_map;             // box {128B worth of columns, 32 rows}, SWIZZLE_128B
  CUtensorMap aux_map;             // same box geometry in AuxT
  CUtensorMap a_half_map;          // cl4: A with a 64-row box (each pair of the cluster fetches half of the shared A tile)
  int cl4;                         // CTA-pair kernels: 1 = clusters of 4 CTAs = two pairs on neighbouring column tiles of the
                                   // same rows; the A tile is fetched once per cluster and multicast to both pairs
  const float* bias;               // [N] or nullptr
  int M, N, K;
  int act;                         // 0 none, 1 exact-erf GELU
  int batch;                       // z tiles (3-D maps) or 1
  int wz_mod;                      // batched W: -1 -> W[z], 0 -> one 2-D W shared by every z, n > 0 -> W[z % n]
  int bias_zstride;                // bias offset per W batch index (wz_mod > 0)
  int tiles_m, tiles_n;
  unsigned long long* trace;       // -DMSMD_GEMM_TRACE builds only: per-role clock64 stamps of the first 16 tiles
};

template <int MODE, int BN_, int EPI_WARPS_, bool HAS_AUX_, typename OutT_, typename AuxT_, bool CTA2_ = false, int OUT_BUFS_ = 2>
struct GemmCfg {
  static constexpr int OUT_BUFS = OUT_BUFS_;   // output staging tiles per epilogue warp = TMA stores in flight + 1
  // CTA2: the tile is 256 x BN on a CTA PAIR (cta_group::2): each CTA holds its 128 rows of A and HALF of the
  // W tile, the leader issues M=256 MMAs that read both shared memories -> 2/3 of the operand bytes per FLOP
  // and 32 KB stages (6 deep) instead of 48 KB (4 deep).
  static constexpr bool CTA2 = CTA2_;
  using OutT = OutT_;
  using AuxT = AuxT_;
  static constexpr int BN = BN_, EPI_WARPS = EPI_WARPS_;
  static constexpr bool HAS_AUX = HAS_AUX_;
  static constexpr int BM = 128;
  static constexpr int ELT = MODE == 1 ? 4 : 2;
  static constexpr int BK = 128 / ELT;  // one 128-byte swizzle atom of K per stage
  static constexpr int UK = 32 / ELT;   // K per tcgen05.mma (32 bytes)
  static constexpr int B_ROWS = CTA2 ? BN / 2 : BN;     // W rows this CTA stages per k-block
  static constexpr int A_BYTES = BM * 128, B_BYTES = B_ROWS * 128;
  static constexpr int UMMA_M = CTA2 ? 256 : 128;
  static constexpr int NSPLIT = (MODE == 0 || MODE == 3) ? 1 : 2;
  static constexpr int STAGE_BYTES = NSPLIT * (A_BYTES + B_BYTES);
  static constexpr int OUT_COLS = 128 / (int)sizeof(OutT);
  static constexpr int AUX_COLS = 128 / (int)sizeof(AuxT);
  static constexpr int EPI_WARP_BYTES = OUT_BUFS * 4096 + (HAS_AUX ? 8192 : 0);  // out staging (+ 2 aux) tiles of 4 KB
  static constexpr int EPI_BYTES = EPI_WARPS * EPI_WARP_BYTES;
  static constexpr int BAR_BYTES = 256 + 2 * 256 * 4;  // mbarriers + TMEM slot, then 2 bias tiles of <= 256 floats
  static constexpr int ALIGN_SLACK = 512;              // dynamic smem base is >= 512-byte aligned in practice; checked
  static constexpr int BUDGET = 227 * 1024 - ALIGN_SLACK - BAR_BYTES;
  static constexpr int STAGES_RAW = (BUDGET - EPI_BYTES) / STAGE_BYTES;
  static constexpr int STAGES = STAGES_RAW > 6 ? 6 : STAGES_RAW;
  static constexpr int SMEM_BYTES = ALIGN_SLACK + STAGES * STAGE_BYTES + EPI_BYTES + BAR_BYTES;
  static constexpr int THREADS = 64 + 32 * EPI_WARPS;
  // MODE 1 keeps the small cross terms (hi*lo + lo*hi) in their own accumulator: the tensor core adds into
  // the accumulator with truncation, so the error grows with the number of MMAs chained on one accumulator.
  static constexpr int ACC_COLS = NSPLIT * BN;  // TMEM columns per accumulator stage
  static constexpr int TMEM_NEED = 2 * ACC_COLS;
  static constexpr int TMEM_COLS = (TMEM_NEED <= 32) ? 32 : (TMEM_NEED <= 64) ? 64 : (TMEM_NEED <= 128) ? 128 : (TMEM_NEED <= 256) ? 256 : 512;
  static constexpr int COL_SPLIT = EPI_WARPS / 4;  // column ranges handled by different epilogue warps
  static constexpr int COLS_PER_WARP = BN / COL_SPLIT;
  static_assert(EPI_WARPS == 4 || EPI_WARPS == 8, "epilogue warps must cover the 4 TMEM lane quarters");
  static_assert(BN % 32 == 0 && BN <= 256 && TMEM_NEED <= 512, "BN");
  static_assert(COLS_PER_WARP % 64 == 0, "the epilogue processes 32-column chunks in pairs");
  static_assert(SMEM_BYTES <= 227 * 1024, "shared memory budget");
  static_assert(STAGES >= 2, "not enough shared memory for a pipeline");
  static_assert(!CTA2 || (MODE != 1 && !HAS_AUX && BN % 32 == 0), "CTA-pair variant: 16-bit operands, no aux");
};

// erf by Abramowitz-Stegun 7.1.26 (|err| <= 1.5e-7): enough for a bf16-rounded GELU, 3x cheaper than erff
__device__ __forceinline__ float erf_fast(float x) {
  const float ax = fabsf(x);
  const float t = __fdividef(1.0f, fmaf(0.3275911f, ax, 1.0f));
  float p = fmaf(1.061405429f, t, -1.453152027f);
  p = fmaf(p, t, 1.421413741f);
  p = fmaf(p, t, -0.284496736f);
  p = fmaf(p, t, 0.254829592f);
  const float r = 1.0f - p * t * __expf(-ax * ax);
  return copysignf(r, x);
}
// exact-erf GELU through the identity Phi(x) = 0.5 (1 + tanh(atanh(erf(x/sqrt2)))): the odd function
// atanh(erf(x/sqrt2)) is fitted by x (a + b x^2 + c x^4) on |x| <= 8 (max |GELU error| 2.5e-5, fitted in
// tools/, 150x below the bf16 rounding of the output), so one MUFU.TANH replaces erf's RCP + EX2:
// 9 instructions per element instead of ~25 - the bf16 GELU epilogue must stay below the 4096-cycle MMA time
// of a 128x256x512 tile.
__device__ __forceinline__ float gelu_tanh3(float x) {
  // the fit holds for |x| <= 8; beyond it x^2 is clamped, so u = x * p(64) = 1.726 x >= 13.8 in magnitude and tanh
  // has long saturated (one FMNMX instead of a two-sided clamp of x)
  const float x2 = fminf(x * x, 64.0f);
  const float u = x * fmaf(x2, fmaf(x2, -0.000351516788570472f, 0.037005646019657945f), 0.7975078842869763f);
  float th;
  asm("tanh.approx.f32 %0, %1;" : "=f"(th) : "f"(u));
  const float hx = 0.5f * x;
  return fmaf(hx, th, hx);
}
template <int MODE>
__device__ __forceinline__ float gelu_erf(float x) {
  if constexpr (MODE == 0) return gelu_tanh3(x);
  else if constexpr (MODE == 3) return 0.5f * x * (1.0f + erf_fast(x * 0.70710678118654752f));   // 1.5e-7: below fp16 rounding
  else return 0.5f * x * (1.0f + erff(x * 0.70710678118654752f));
}
template <class T> struct is_half_t { static constexpr bool value = false; };
template <> struct is_half_t<__half> { static constexpr bool value = true; };
// two floats -> one packed 16-bit pair in the storage format of T (bf16 or fp16)
template <class T>
__device__ __forceinline__ uint32_t pack16x2(float a, float b) {
  if constexpr (is_half_t<T>::value) {
    __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
  } else {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
  }
}
template <class T>
__device__ __forceinline__ float2 unpack16x2(uint32_t w) {
  if constexpr (is_half_t<T>::value) return __half22float2(*reinterpret_cast<const __half2*>(&w));
  else return make_float2(__uint_as_float(w << 16), __uint_as_float(w & 0xffff0000u));
}

// Per-role timeline of the first 16 tiles (clock64 stamps), compiled in only with -DMSMD_GEMM_TRACE (tools/pair_probe.py)
__device__ __forceinline__ void trace_stamp(unsigned long long* tr, int role, int it, int ev) {
#ifdef MSMD_GEMM_TRACE
  if (tr != nullptr && it < 16) tr[((blockIdx.x * 3 + role) * 16 + it) * 4 + ev] = clock64();
#endif
}

template <class Cfg, int MODE, bool GELU>
__global__ void __launch_bounds__(Cfg::THREADS, 1) gemm_tc_kernel(const __grid_constant__ GemmParams p) {
  using namespace tc;
  using OutT = typename Cfg::OutT;
  using AuxT = typename Cfg::AuxT;
  constexpr int BM = Cfg::BM, BN = Cfg::BN, BK = Cfg::BK, STAGES = Cfg::STAGES;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* stage_base = smem;
  uint8_t* epi_base = smem + STAGES * Cfg::STAGE_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(epi_base + Cfg::EPI_BYTES);
  uint64_t* full_bar = bars;                    // [STAGES]
  uint64_t* empty_bar = bars + STAGES;          // [STAGES]
  uint64_t* tfull_bar = bars + 2 * STAGES;      // [2]
  uint64_t* tempty_bar = bars + 2 * STAGES + 2; // [2]
  uint64_t* aux_bar = bars + 2 * STAGES + 4;    // [EPI_WARPS][2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4 + 2 * Cfg::EPI_WARPS);
  float* bias_tile = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(bars) + 256);  // [2][BN]
  static_assert((2 * Cfg::STAGES + 4 + 2 * Cfg::EPI_WARPS) * 8 + 4 <= 256, "barrier block overflows its 256 bytes");
  if (threadIdx.x == 0 && reinterpret_cast<uint8_t*>(bias_tile) + 2 * 256 * 4 > smem_raw + Cfg::SMEM_BYTES) __trap();

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int crank = Cfg::CTA2 ? (int)cluster_ctarank() : 0;   // rank in the cluster (2 CTAs, or 4 = two pairs when p.cl4)
  const int cta_rank = crank & 1;                             // rank in the CTA pair
  const bool cl4 = Cfg::CTA2 && p.cl4 != 0;
  const uint16_t pair_mask = (uint16_t)(3u << (crank & ~1)); // the two CTAs of this pair, as cluster ranks
  const int tile0 = Cfg::CTA2 ? (int)blockIdx.x / 2 : (int)blockIdx.x;       // first tile of this CTA (pair)
  const int tstride = Cfg::CTA2 ? (int)gridDim.x / 2 : (int)gridDim.x;
  const int num_tiles = p.tiles_m * p.tiles_n * p.batch;
  const int num_kb = (p.K + BK - 1) / BK;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&p.a_map);
    prefetch_tmap(&p.b_map);
    prefetch_tmap(&p.out_map);
    if (Cfg::NSPLIT == 2) { prefetch_tmap(&p.a_lo_map); prefetch_tmap(&p.b_lo_map); }
    if (cl4) prefetch_tmap(&p.a_half_map);
    if (Cfg::HAS_AUX) prefetch_tmap(&p.aux_map);
    // cl4: a slot is written by this pair AND (the shared A half) by the sibling pair: it is free when both pairs' MMAs retired
    for (int s = 0; s < STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], cl4 ? 2 : 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(&tfull_bar[a], 1); mbar_init(&tempty_bar[a], Cfg::EPI_WARPS * (Cfg::CTA2 ? 2 : 1)); }
    for (int i = 0; i < 2 * Cfg::EPI_WARPS; ++i) mbar_init(&aux_bar[i], 1);
    fence_barrier_init();
  }
  if (warp == 1) {
    if constexpr (Cfg::CTA2) tmem_alloc_2sm(tmem_slot, Cfg::TMEM_COLS);
    else tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
  }
  tc_fence_before();
  if constexpr (Cfg::CTA2) cluster_sync();  // the peer's barriers are initialised before anyone signals them
  else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  auto tile_coords = [&](int t, int& m0, int& n0, int& z) {
    const int per_z = p.tiles_m * p.tiles_n;
    z = t / per_z;
    const int r = t - z * per_z;
    m0 = (r / p.tiles_n) * (Cfg::CTA2 ? 2 * BM : BM) + cta_rank * BM;
    n0 = (r % p.tiles_n) * BN;
  };

  if (warp == 0) {
    // ------------------------------------------------ TMA producer (lane 0 issues; the warp stays converged)
    int s = 0;
    uint32_t ph = 0;
    int pit = 0;
    for (int t = tile0; t < num_tiles; t += tstride, ++pit) {
      int m0, n0, z;
      tile_coords(t, m0, n0, z);
      for (int kb = 0; kb < num_kb; ++kb) {
        if (lane == 0) {
          if (kb == 0) trace_stamp(p.trace, 0, pit, 0);
          mbar_wait(&empty_bar[s], ph ^ 1);
          if (kb == 0) trace_stamp(p.trace, 0, pit, 1);
          if (kb == num_kb - 1) trace_stamp(p.trace, 0, pit, 2);
          uint8_t* sa = stage_base + s * Cfg::STAGE_BYTES;
          uint8_t* sb = sa + Cfg::NSPLIT * Cfg::A_BYTES;
          if constexpr (Cfg::CTA2) {
            if (cta_rank == 0) mbar_expect_tx(&full_bar[s], 2 * Cfg::STAGE_BYTES);  // both CTAs' boxes land here
            if (cl4) {   // rows [64j, 64j+64) of this CTA's A half, j = pair index: written here AND in the sibling pair's CTA
              const int j = crank >> 1;
              tma_load_2d_2sm_mc(sa + j * (Cfg::A_BYTES / 2), &p.a_half_map, &full_bar[s], kb * BK, m0 + j * (BM / 2),
                                 (uint16_t)(5u << cta_rank));
            } else {
              tma_load_2d_2sm(sa, &p.a_map, &full_bar[s], kb * BK, m0);
            }
            tma_load_2d_2sm(sb, &p.b_map, &full_bar[s], kb * BK, n0 + cta_rank * Cfg::B_ROWS);
            if (Cfg::NSPLIT == 2) {
              tma_load_2d_2sm(sa + Cfg::A_BYTES, &p.a_lo_map, &full_bar[s], kb * BK, m0);
              tma_load_2d_2sm(sb + Cfg::B_BYTES, &p.b_lo_map, &full_bar[s], kb * BK, n0 + cta_rank * Cfg::B_ROWS);
            }
          } else if (p.batch > 1) {
            mbar_expect_tx(&full_bar[s], Cfg::STAGE_BYTES);
            tma_load_3d(sa, &p.a_map, &full_bar[s], kb * BK, m0, z);
            if (p.wz_mod == 0) tma_load_2d(sb, &p.b_map, &full_bar[s], kb * BK, n0);
            else tma_load_3d(sb, &p.b_map, &full_bar[s], kb * BK, n0, p.wz_mod > 0 ? z % p.wz_mod : z);
          } else {
            mbar_expect_tx(&full_bar[s], Cfg::STAGE_BYTES);
            tma_load_2d(sa, &p.a_map, &full_bar[s], kb * BK, m0);
            tma_load_2d(sb, &p.b_map, &full_bar[s], kb * BK, n0);
            if (Cfg::NSPLIT == 2) {
              tma_load_2d(sa + Cfg::A_BYTES, &p.a_lo_map, &full_bar[s], kb * BK, m0);
              tma_load_2d(sb + Cfg::B_BYTES, &p.b_lo_map, &full_bar[s], kb * BK, n0);
            }
          }
        }
        __syncwarp();
        if (++s == STAGES) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------ MMA issuer (lane 0 issues for the whole CTA)
    constexpr uint32_t idesc = make_idesc(MODE == 0 ? 1 : (MODE == 1 ? 2 : 0), Cfg::UMMA_M, BN);   // bf16 / tf32 / fp16
    int s = 0;
    uint32_t ph = 0;
    int it = 0;
    for (int t = (Cfg::CTA2 && cta_rank != 0) ? num_tiles : tile0; t < num_tiles; t += tstride, ++it) {  // leader only
      const int a = it & 1;
      const uint32_t aph = (it >> 1) & 1;
      const uint32_t d_tmem = tmem_base + a * Cfg::ACC_COLS;
      if (lane == 0) {
        trace_stamp(p.trace, 1, it, 0);
        mbar_wait(&tempty_bar[a], aph ^ 1);
        tc_fence_after();
        trace_stamp(p.trace, 1, it, 1);
      }
      __syncwarp();
      for (int kb = 0; kb < num_kb; ++kb) {
        if (lane == 0) {
          mbar_wait(&full_bar[s], ph);
          tc_fence_after();
          if (kb == 0) trace_stamp(p.trace, 1, it, 2);
          const uint32_t sa = smem_u32(stage_base + s * Cfg::STAGE_BYTES);
          const uint32_t sb = sa + Cfg::NSPLIT * Cfg::A_BYTES;
          const uint64_t da = make_smem_desc_sw128(sa), db = make_smem_desc_sw128(sb);
#pragma unroll
          for (int k = 0; k < BK / Cfg::UK; ++k) {
            const uint32_t acc = (kb | k) != 0;
            if constexpr (Cfg::NSPLIT == 1) {
              if constexpr (Cfg::CTA2) umma_2sm(d_tmem, desc_advance(da, k * 32), desc_advance(db, k * 32), idesc, acc);
              else umma<0>(d_tmem, desc_advance(da, k * 32), desc_advance(db, k * 32), idesc, acc);
            } else {
              const uint64_t dal = make_smem_desc_sw128(sa + Cfg::A_BYTES), dbl = make_smem_desc_sw128(sb + Cfg::B_BYTES);
              constexpr int KIND = MODE == 1 ? 1 : 0;
              if constexpr (Cfg::CTA2) {
                umma_2sm(d_tmem + BN, desc_advance(dal, k * 32), desc_advance(db, k * 32), idesc, acc);  // lo * hi
                umma_2sm(d_tmem + BN, desc_advance(da, k * 32), desc_advance(dbl, k * 32), idesc, 1u);   // hi * lo
                umma_2sm(d_tmem, desc_advance(da, k * 32), desc_advance(db, k * 32), idesc, acc);        // hi * hi
              } else {
                umma<KIND>(d_tmem + BN, desc_advance(dal, k * 32), desc_advance(db, k * 32), idesc, acc);  // lo * hi
                umma<KIND>(d_tmem + BN, desc_advance(da, k * 32), desc_advance(dbl, k * 32), idesc, 1u);   // hi * lo
                umma<KIND>(d_tmem, desc_advance(da, k * 32), desc_advance(db, k * 32), idesc, acc);        // hi * hi
              }
            }
          }
          if constexpr (Cfg::CTA2) umma_commit_2sm(&empty_bar[s], cl4 ? (uint16_t)0xF : pair_mask);
          else umma_commit(&empty_bar[s]);  // smem slot reusable once these MMAs have read it
        }
        __syncwarp();
        if (++s == STAGES) { s = 0; ph ^= 1; }
      }
      if (lane == 0) trace_stamp(p.trace, 1, it, 3);
      if (lane == 0) {  // accumulator complete -> epilogue (of both CTAs in pair mode)
        if constexpr (Cfg::CTA2) umma_commit_2sm(&tfull_bar[a], pair_mask);
        else umma_commit(&tfull_bar[a]);
      }
      __syncwarp();
    }
  } else {
    // ------------------------------------------------ epilogue warps
    const int e = warp - 2;
    const int q = warp & 3;                 // TMEM lane quarter this warp may access
    const int csplit = e / 4;               // which column range of the tile
    uint8_t* my = epi_base + e * Cfg::EPI_WARP_BYTES;
    uint8_t* out_stage = my;                // 2 x [32 rows][128 B], SW128
    uint8_t* aux_stage = my + Cfg::OUT_BUFS * 4096;  // 2 x [32 rows][128 B]
    uint64_t* my_aux_bar = aux_bar + 2 * e;
    constexpr int CPW = Cfg::COLS_PER_WARP;
    constexpr int AUX_PER_TILE = Cfg::HAS_AUX ? CPW / Cfg::AUX_COLS : 1;
    constexpr int EPI_THREADS = 32 * Cfg::EPI_WARPS;
    const int swz = lane & 7;
    const int etid = threadIdx.x - 64;

    auto issue_aux = [&](int f) {  // flat aux-chunk index over this CTA's tiles
      if constexpr (Cfg::HAS_AUX) {
        const int lt = f / AUX_PER_TILE, ck = f % AUX_PER_TILE;
        const int t = tile0 + lt * tstride;
        if (t < num_tiles && lane == 0) {
          int m0, n0, z;
          tile_coords(t, m0, n0, z);
          const int b = f & 1;
          mbar_expect_tx(&my_aux_bar[b], 4096);
          const int c0 = n0 + csplit * CPW + ck * Cfg::AUX_COLS;
          if (p.batch > 1) tma_load_3d(aux_stage + b * 4096, &p.aux_map, &my_aux_bar[b], c0, m0 + q * 32, z);
          else tma_load_2d(aux_stage + b * 4096, &p.aux_map, &my_aux_bar[b], c0, m0 + q * 32);
        }
      }
    };
    int af = 0;        // next aux chunk to consume
    int so = 0;        // output staging buffers written so far (alternates between the two)
    issue_aux(0);

    // bias values of the NEXT tile travel in registers while the current tile is processed (their global-load
    // latency would otherwise sit at the head of every tile's epilogue)
    constexpr int BPT = (BN + EPI_THREADS - 1) / EPI_THREADS;
    float bnext[BPT];
    auto fetch_bias = [&](int t) {
      if (t < num_tiles) {
        int m0, n0, z;
        tile_coords(t, m0, n0, z);
        const float* bias_z = p.bias + (p.wz_mod > 0 ? (z % p.wz_mod) * p.bias_zstride : 0);
#pragma unroll
        for (int i = 0; i < BPT; ++i) {
          const int col = etid + i * EPI_THREADS;
          bnext[i] = (p.bias != nullptr && col < BN && n0 + col < p.N) ? __ldg(bias_z + n0 + col) : 0.f;
        }
      }
    };
    fetch_bias(tile0);

    int it = 0;
    for (int t = tile0; t < num_tiles; t += tstride, ++it) {
      int m0, n0, z;
      tile_coords(t, m0, n0, z);
      const int a = it & 1;
      const uint32_t aph = (it >> 1) & 1;
      // bias tile -> shared (double-buffered by tile parity).  The named barrier also keeps the epilogue warps
      // within one tile of each other, which is what makes reusing buffer `a` two tiles later safe.
      float* sb = bias_tile + a * BN;
#pragma unroll
      for (int i = 0; i < BPT; ++i) {
        const int col = etid + i * EPI_THREADS;
        if (col < BN) sb[col] = bnext[i];
      }
      asm volatile("bar.sync 1, %0;" ::"n"(EPI_THREADS) : "memory");
      fetch_bias(t + tstride);
      if (e == 0 && lane == 0) trace_stamp(p.trace, 2, it, 0);
      mbar_wait(&tfull_bar[a], aph);
      tc_fence_after();
      if (e == 0 && lane == 0) trace_stamp(p.trace, 2, it, 1);
      const uint32_t t_addr = tmem_base + ((uint32_t)(q * 32) << 16) + a * Cfg::ACC_COLS + csplit * CPW;
      const float* sbw = sb + csplit * CPW;

      auto process = [&](uint32_t (&raw)[32], uint32_t (&raw2)[Cfg::NSPLIT == 2 ? 32 : 1], int c) {
        const uint8_t* aux_buf = nullptr;
        int aux_off = 0;
        if constexpr (Cfg::HAS_AUX) {
          if (c % Cfg::AUX_COLS == 0) {
            __syncwarp();               // every lane is done with the buffer the prefetch will overwrite
            issue_aux(af + 1);
            mbar_wait(&my_aux_bar[af & 1], (af >> 1) & 1);
          }
          aux_buf = aux_stage + (af & 1) * 4096 + lane * 128;
          aux_off = (c % Cfg::AUX_COLS) * (int)sizeof(AuxT) / 16;  // first 16-byte chunk of this 32-col slice
        }
        float v[32];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float4 b4 = *reinterpret_cast<const float4*>(sbw + c + 4 * j);   // broadcast LDS.128
          v[4 * j + 0] = __uint_as_float(raw[4 * j + 0]) + b4.x;
          v[4 * j + 1] = __uint_as_float(raw[4 * j + 1]) + b4.y;
          v[4 * j + 2] = __uint_as_float(raw[4 * j + 2]) + b4.z;
          v[4 * j + 3] = __uint_as_float(raw[4 * j + 3]) + b4.w;
        }
        if constexpr (MODE == 1) {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] += __uint_as_float(raw2[j]);
        }
        if constexpr (MODE == 2) {   // cross terms carry the 2^11 scale of the residual operands
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = fmaf(__uint_as_float(raw2[j]), 1.0f / 2048.0f, v[j]);
        }
        if constexpr (GELU) {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = gelu_erf<MODE>(v[j]);
        }
        if constexpr (Cfg::HAS_AUX) {
          if constexpr (sizeof(AuxT) == 4) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float4 r4 = *reinterpret_cast<const float4*>(aux_buf + (((aux_off + j) ^ swz) << 4));
              v[4 * j + 0] += r4.x; v[4 * j + 1] += r4.y; v[4 * j + 2] += r4.z; v[4 * j + 3] += r4.w;
            }
          } else {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const uint4 r4 = *reinterpret_cast<const uint4*>(aux_buf + (((aux_off + j) ^ swz) << 4));
              const uint32_t w[4] = {r4.x, r4.y, r4.z, r4.w};
#pragma unroll
              for (int u = 0; u < 4; ++u) {
                const float2 f2 = unpack16x2<AuxT>(w[u]);
                v[8 * j + 2 * u + 0] += f2.x;
                v[8 * j + 2 * u + 1] += f2.y;
              }
            }
          }
          if ((c + 32) % Cfg::AUX_COLS == 0) ++af;
        }
        // ---- registers -> swizzled staging (two buffers) -> TMA store
        const int o_off = (c % Cfg::OUT_COLS) * (int)sizeof(OutT) / 16;
        if (c % Cfg::OUT_COLS == 0) {
          if (lane == 0) tma_store_wait_read<Cfg::OUT_BUFS - 1>();  // the store that last used this buffer has finished reading it
          __syncwarp();
        }
        uint8_t* obuf = out_stage + (so % Cfg::OUT_BUFS) * 4096;
        uint8_t* orow = obuf + lane * 128;
        if constexpr (sizeof(OutT) == 4) {
#pragma unroll
          for (int j = 0; j < 8; ++j)
            *reinterpret_cast<float4*>(orow + (((o_off + j) ^ swz) << 4)) =
                make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            uint32_t w[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) w[u] = pack16x2<OutT>(v[8 * j + 2 * u], v[8 * j + 2 * u + 1]);
            *reinterpret_cast<uint4*>(orow + (((o_off + j) ^ swz) << 4)) = make_uint4(w[0], w[1], w[2], w[3]);
          }
        }
        if ((c + 32) % Cfg::OUT_COLS == 0) {
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            const int c0 = n0 + csplit * CPW + (c / Cfg::OUT_COLS) * Cfg::OUT_COLS;
            if (p.batch > 1) tma_store_3d(&p.out_map, obuf, c0, m0 + q * 32, z);
            else tma_store_2d(&p.out_map, obuf, c0, m0 + q * 32);
            tma_store_commit();
          }
          ++so;
        }
      };

      auto release_acc = [&]() {   // every TMEM read of this tile has landed in registers: hand the accumulator back
        if (e == 0 && lane == 0) trace_stamp(p.trace, 2, it, 2);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (Cfg::CTA2 && cta_rank != 0) mbar_arrive_cluster(&tempty_bar[a], crank & ~1);  // the leader's MMA warp waits for both
          else mbar_arrive(&tempty_bar[a]);
        }
      };
      if constexpr (Cfg::NSPLIT == 2) {
        // software-pipelined TMEM reads: chunk c+1 is in flight while chunk c is processed
        uint32_t rA[32], rB[32], rA2[32], rB2[32];
        tmem_ld32(t_addr, rA);
        tmem_ld32(t_addr + BN, rA2);
#pragma unroll 1
        for (int c = 0; c < CPW; c += 64) {
          tmem_ld_wait();
          tmem_ld32(t_addr + c + 32, rB);
          tmem_ld32(t_addr + BN + c + 32, rB2);
          process(rA, rA2, c);
          tmem_ld_wait();
          if (c + 64 < CPW) {
            tmem_ld32(t_addr + c + 64, rA);
            tmem_ld32(t_addr + BN + c + 64, rA2);
          } else {
            release_acc();
          }
          process(rB, rB2, c + 32);
        }
      } else {
        // 64 columns (two 32-column loads) in flight while the previous 64 are processed
        uint32_t r0[32], r1[32], r2[32], r3[32];
        uint32_t none[1];
        tmem_ld32(t_addr, r0);
        tmem_ld32(t_addr + 32, r1);
#pragma unroll 1
        for (int c = 0; c < CPW; c += 128) {
          tmem_ld_wait();
          const bool more = c + 64 < CPW;
          if (more) {
            tmem_ld32(t_addr + c + 64, r2);
            tmem_ld32(t_addr + c + 96, r3);
          } else {
            release_acc();
          }
          process(r0, none, c);
          process(r1, none, c + 32);
          if (more) {
            tmem_ld_wait();
            if (c + 128 < CPW) {
              tmem_ld32(t_addr + c + 128, r0);
              tmem_ld32(t_addr + c + 160, r1);
            } else {
              release_acc();
            }
            process(r2, none, c + 64);
            process(r3, none, c + 96);
          }
        }
      }
      if (e == 0 && lane == 0) trace_stamp(p.trace, 2, it, 3);
    }
    if (lane == 0) tma_store_wait<0>();
  }

  tc_fence_before();
  if constexpr (Cfg::CTA2) cluster_sync();  // the peer may still be reading this CTA's smem / signalling its barriers
  else __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    if constexpr (Cfg::CTA2) tmem_dealloc_2sm(tmem_base, Cfg::TMEM_COLS);
    else tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
  }
}

// ---------------------------------------------------------------------------------------------
// Host-side description of one GEMM call.  Element strides; row-major [rows, K] operands.
struct GemmDesc {
  int mode = 0;                 // 0 bf16, 1 tf32x3, 2 fp16x3 (A/W hi and lo are __half, x = hi + 2^-11 lo), 3 fp16 one pass
  const void* A = nullptr;      // [M,K] bf16 (mode 0) / fp32 hi (mode 1)
  const void* A_lo = nullptr;   // mode 1
  const void* W = nullptr;      // [N,K]
  const void* W_lo = nullptr;   // mode 1
  const float* bias = nullptr;  // [N]
  const void* aux = nullptr;    // [M,N] residual added after bias/activation
  void* out = nullptr;          // [M,N]
  int M = 0, N = 0, K = 0;
  int64_t lda = 0, ldw = 0, ldo = 0, ld_aux = 0;  // row strides (elements)
  int out_f32 = 0, aux_f32 = 0;
  int act = 0;
  // optional batch (z) dimension: strides in elements; batch<=1 means plain 2-D
  int batch = 1;
  int64_t sA = 0, sW = 0, sO = 0, sAux = 0;
  int wz_mod = -1;              // see GemmParams (only read when batch > 1)
  int bias_zstride = 0;
  int gelu_heavy = 0;           // use 8 epilogue warps
};

int gemm_tc_launch(const GemmDesc& d, cudaStream_t st);
// `overflow` (optional, device): set to 1 when a value lies outside the fp16 range, which the split cannot represent
int split_f16(const float* x, __half* hi, __half* lo, int64_t n, cudaStream_t st, int* overflow = nullptr);

}  // namespace msmd
