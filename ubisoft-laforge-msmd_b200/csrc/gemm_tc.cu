// Host side of the tcgen05 GEMM core: tensor-map construction, config dispatch, C-ABI test entry.
#include "gemm_tc.cuh"
#include "profile.cuh"
#include <cuda_fp16.h>
#include <algorithm>
#include <cudaTypedefs.h>
#include <mutex>
#include <cstdlib>
#include <cstring>
#include <vector>

namespace msmd {

static PFN_cuTensorMapEncodeTiled_v12000 get_encode() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(p);
  });
  return fn;
}

int make_tmap(CUtensorMap* out, const void* base, CUtensorMapDataType dt, int rank, const uint64_t* dims,
              const uint64_t* strides_bytes, const uint32_t* box, CUtensorMapSwizzle swz) {
  auto enc = get_encode();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled entry point unavailable (driver too old?)");
    return MSMD_ERR_CUDA;
  }
  cuuint64_t gdim[5], gstr[4];
  cuuint32_t bx[5], es[5];
  for (int i = 0; i < rank; ++i) { gdim[i] = dims[i]; bx[i] = box[i]; es[i] = 1; }
  for (int i = 0; i + 1 < rank; ++i) gstr[i] = strides_bytes[i];
  if ((reinterpret_cast<uintptr_t>(base) & 15) != 0) {
    set_error("tensor map: base address %p is not 16-byte aligned", base);
    return MSMD_ERR_INVALID;
  }
  for (int i = 0; i + 1 < rank; ++i)
    if (gstr[i] % 16 != 0) {
      set_error("tensor map: stride %llu bytes is not a multiple of 16", (unsigned long long)gstr[i]);
      return MSMD_ERR_INVALID;
    }
  CUresult r = enc(out, dt, rank, const_cast<void*>(base), gdim, gstr, bx, es, CU_TENSOR_MAP_INTERLEAVE_NONE, swz,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with CUresult %d (rank %d dims %llu,%llu box %u,%u)", (int)r, rank,
              (unsigned long long)gdim[0], (unsigned long long)(rank > 1 ? gdim[1] : 0), bx[0], rank > 1 ? bx[1] : 0);
    return MSMD_ERR_CUDA;
  }
  return MSMD_OK;
}

int make_tmap_2d(CUtensorMap* out, const void* base, CUtensorMapDataType dt, uint64_t inner, uint64_t outer,
                 uint64_t row_stride_bytes, uint32_t box_inner, uint32_t box_outer, CUtensorMapSwizzle swz) {
  uint64_t dims[2] = {inner, outer};
  uint64_t str[1] = {row_stride_bytes};
  uint32_t box[2] = {box_inner, box_outer};
  return make_tmap(out, base, dt, 2, dims, str, box, swz);
}

static int make_tmap_23(CUtensorMap* out, const void* base, CUtensorMapDataType dt, int esz, uint64_t inner,
                        uint64_t outer, int64_t row_stride, int batch, int64_t batch_stride, uint32_t box_inner,
                        uint32_t box_outer) {
  if (batch <= 1)
    return make_tmap_2d(out, base, dt, inner, outer, (uint64_t)row_stride * esz, box_inner, box_outer,
                        CU_TENSOR_MAP_SWIZZLE_128B);
  uint64_t dims[3] = {inner, outer, (uint64_t)batch};
  uint64_t str[2] = {(uint64_t)row_stride * esz, (uint64_t)batch_stride * esz};
  uint32_t box[3] = {box_inner, box_outer, 1};
  return make_tmap(out, base, dt, 3, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B);
}

template <class Cfg, int MODE, bool GELU>
static int launch_cfg2(const GemmDesc& d, cudaStream_t st) {
  GemmParams p;
  memset(&p, 0, sizeof(p));
  const auto in_dt = MODE == 0 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16
                               : (MODE == 1 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16);
  const int esz = Cfg::ELT;
  int rc;
  if ((rc = make_tmap_23(&p.a_map, d.A, in_dt, esz, d.K, d.M, d.lda, d.batch, d.sA, Cfg::BK, Cfg::BM))) return rc;
  {
    const int wb = (d.batch > 1 && d.wz_mod != 0) ? (d.wz_mod > 0 ? d.wz_mod : d.batch) : 1;
    if ((rc = make_tmap_23(&p.b_map, d.W, in_dt, esz, d.K, d.N, d.ldw, wb, d.sW, Cfg::BK, Cfg::B_ROWS))) return rc;
  }
  if (Cfg::NSPLIT == 2) {
    MSMD_REQUIRE(d.A_lo && d.W_lo, "gemm: the three-pass modes need the lo operands");
    MSMD_REQUIRE(d.batch <= 1, "gemm: batched three-pass GEMMs are not implemented");
    if ((rc = make_tmap_23(&p.a_lo_map, d.A_lo, in_dt, esz, d.K, d.M, d.lda, 1, 0, Cfg::BK, Cfg::BM))) return rc;
    if ((rc = make_tmap_23(&p.b_lo_map, d.W_lo, in_dt, esz, d.K, d.N, d.ldw, 1, 0, Cfg::BK, Cfg::B_ROWS))) return rc;
  }
  using OutT = typename Cfg::OutT;
  using AuxT = typename Cfg::AuxT;
  const auto dt16 = MODE == 3 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  const auto out_dt = sizeof(OutT) == 2 ? dt16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
  if ((rc = make_tmap_23(&p.out_map, d.out, out_dt, sizeof(OutT), d.N, d.M, d.ldo, d.batch, d.sO, Cfg::OUT_COLS, 32)))
    return rc;
  if (Cfg::HAS_AUX) {
    const auto aux_dt = sizeof(AuxT) == 2 ? dt16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
    if ((rc = make_tmap_23(&p.aux_map, d.aux, aux_dt, sizeof(AuxT), d.N, d.M, d.ld_aux, d.batch, d.sAux,
                           Cfg::AUX_COLS, 32)))
      return rc;
  }
  p.bias = d.bias;
  p.M = d.M; p.N = d.N; p.K = d.K;
  p.act = d.act;
  p.batch = d.batch < 1 ? 1 : d.batch;
  p.wz_mod = d.wz_mod;
  p.bias_zstride = d.bias_zstride;
#ifdef MSMD_GEMM_TRACE
  static const bool env_trace = getenv("MSMD_GEMM_TRACE") != nullptr;
#else
  constexpr bool env_trace = false;
#endif
  static unsigned long long* trace_buf = nullptr;
  constexpr size_t kTraceN = (size_t)kNumSMs * 3 * 16 * 4;
  if (env_trace) {
    if (!trace_buf) MSMD_CHECK_CUDA(cudaMalloc(&trace_buf, kTraceN * 8));
    MSMD_CHECK_CUDA(cudaMemsetAsync(trace_buf, 0, kTraceN * 8, st));
    p.trace = trace_buf;
  }
  p.tiles_m = cdiv(d.M, Cfg::CTA2 ? 2 * Cfg::BM : Cfg::BM);
  p.tiles_n = cdiv(d.N, Cfg::BN);
  const int tiles = p.tiles_m * p.tiles_n * p.batch;
  auto kern = gemm_tc_kernel<Cfg, MODE, GELU>;
  static bool attr_set = false;  // per template instantiation
  if (!attr_set) {
    MSMD_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
    attr_set = true;
  }
  ProfileScope prof(MODE == 0 ? "gemm_bf16" : (MODE == 1 ? "gemm_tf32x3" : (MODE == 2 ? "gemm_fp16x3" : "gemm_fp16")), st);
  char shape_name[64];
  snprintf(shape_name, sizeof(shape_name), "gemm_%dx%dx%d%s", d.M, d.N, d.K, Cfg::CTA2 ? "_pair" : "");
  ProfileScope prof2(profiling_on() ? strdup(shape_name) : "", st);
  if constexpr (Cfg::CTA2) {
    int pairs = tiles < kNumSMs / 2 ? tiles : kNumSMs / 2;
    cudaLaunchConfig_t cfg = {};
    cfg.blockDim = dim3(Cfg::THREADS);
    cfg.dynamicSmemBytes = Cfg::SMEM_BYTES;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    // Clusters of 4 = two pairs on neighbouring column tiles of the same rows, the A tile fetched once and multicast
    // (default).  Bit-identical results, -1.1% per sampling step on one box: the L2 reads
    // drop by a quarter but the main loop is bound on the SM side (TMA fill 64 B/clk + MMA operand reads 64 B/clk +
    // epilogue staging against 128 B/clk of shared-memory bandwidth at MMA peak), not by L2.  Needs an even number of
    // column tiles (both pairs of a cluster then always have a tile) and enough co-resident 4-CTA clusters that no
    // round is added to the persistent schedule.
    if (Cfg::NSPLIT == 1 && p.tiles_n % 2 == 0 && tiles >= 4) {
      static int max_cl4 = -1;     // per instantiation
      if (max_cl4 < 0) {
        cfg.gridDim = dim3(kNumSMs / 4 * 4);
        attr[0].val.clusterDim.x = 4;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        int nc = 0;
        if (cudaOccupancyMaxActiveClusters(&nc, kern, &cfg) != cudaSuccess) { (void)cudaGetLastError(); nc = 0; }
        max_cl4 = nc < kNumSMs / 4 ? nc : kNumSMs / 4;
        attr[0].val.clusterDim.x = 2;
      }
      const int want = pairs / 2;                                          // clusters the 2-CTA schedule would occupy
      const int cl = want < max_cl4 ? want : max_cl4;
      if (cl >= 1 && cdiv(tiles, 2 * cl) <= cdiv(tiles, pairs)) {          // no extra round
        if (make_tmap_23(&p.a_half_map, d.A, in_dt, esz, d.K, d.M, d.lda, 1, 0, Cfg::BK, Cfg::BM / 2)) return MSMD_ERR_CUDA;
        p.cl4 = 1;
        pairs = 2 * cl;
        attr[0].val.clusterDim.x = 4;
      }
    }
    cfg.gridDim = dim3(2 * pairs);
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    MSMD_CHECK_CUDA(cudaLaunchKernelEx(&cfg, kern, p));
  } else {
    const int grid = tiles < kNumSMs ? tiles : kNumSMs;
    kern<<<grid, Cfg::THREADS, Cfg::SMEM_BYTES, st>>>(p);
  }
  MSMD_CHECK_LAUNCH();
  if (env_trace) {
    static int dumps = 0;
    std::vector<unsigned long long> h(kTraceN);
    MSMD_CHECK_CUDA(cudaStreamSynchronize(st));
    MSMD_CHECK_CUDA(cudaMemcpy(h.data(), trace_buf, kTraceN * 8, cudaMemcpyDeviceToHost));
    if (dumps++ % 23 == 22) {   // one warm launch per shape in tools/pair_probe.py
      for (int cta : {0, 1, 77}) {
        const unsigned long long t0 = h[((size_t)cta * 3 + 0) * 64 + 0];
        fprintf(stderr, "[trace] %s cta %d (cycles since the producer's first stamp)\n", shape_name, cta);
        const char* names[3] = {"tma  [start, slot0 free, last kb issued, -]", "mma  [start, acc free, first full, last issued]",
                                "epi0 [start, acc full, tmem drained, done]"};
        for (int role = 0; role < 3; ++role) {
          fprintf(stderr, "  %s\n", names[role]);
          for (int it = 0; it < 12; ++it) {
            const unsigned long long* e = &h[(((size_t)cta * 3 + role) * 16 + it) * 4];
            if (!e[0] && !e[1]) break;
            fprintf(stderr, "    tile %2d: %7lld %7lld %7lld %7lld\n", it, (long long)(e[0] - t0), (long long)(e[1] - t0),
                    (long long)(e[2] ? e[2] - t0 : 0), (long long)(e[3] ? e[3] - t0 : 0));
          }
        }
      }
    }
  }
  return MSMD_OK;
}

template <class Cfg, int MODE>
static int launch_cfg(const GemmDesc& d, cudaStream_t st) {
  return d.act ? launch_cfg2<Cfg, MODE, true>(d, st) : launch_cfg2<Cfg, MODE, false>(d, st);
}

// single-pass 16-bit GEMMs: MODE 0 (bf16 storage) and MODE 3 (fp16 storage) share every tile configuration
template <int MODE, class H>
static int dispatch16(const GemmDesc& d, cudaStream_t st) {
  const bool aux = d.aux != nullptr;
  // narrow outputs (N <= 128) use the 128-wide tile so small problems still spread over SMs
  const bool narrow = d.N <= 128;
  // measured on B200 (tools/pair_probe.py, M = 21312): the single-CTA 128x256 tile needs 96 B/clk of operands per SM
  // at MMA peak and the L2->SM path delivers ~60, so its main loop runs at ~1.3 PFLOP/s; the pair (64 B/clk) is
  // MMA-bound.  Pair vs single: 1536x512 31.8/33.5 us, 2048x512+GELU 50.0/53.2, 512x2048 41.4/46.1, 512x512 tie.
  const bool pair = !aux && !d.out_f32 && d.batch <= 1 && d.N >= 256 && d.M >= 2048;
  const bool epi8 = d.gelu_heavy != 0;
  if (pair) {
    if (epi8) return launch_cfg<GemmCfg<MODE, 256, 8, false, H, H, true>, MODE>(d, st);
    return launch_cfg<GemmCfg<MODE, 256, 4, false, H, H, true>, MODE>(d, st);
  }
  // a handful of rows (the person-token projections, M = sequences): 64-wide tiles spread the N dimension over
  // 4x more SMs, and the whole K extent of a tile fits the 6-stage ring, so one TMA latency covers it
  if (!aux && !d.out_f32 && d.batch <= 1 && d.M <= 512 && d.N >= 256)
    return launch_cfg<GemmCfg<MODE, 64, 4, false, H, H>, MODE>(d, st);
  if (!aux) {
    if (d.out_f32) {
      return narrow ? launch_cfg<GemmCfg<MODE, 128, 4, false, float, float>, MODE>(d, st)
                    : launch_cfg<GemmCfg<MODE, 256, 4, false, float, float>, MODE>(d, st);
    }
    if (epi8 && !narrow) return launch_cfg<GemmCfg<MODE, 256, 8, false, H, H>, MODE>(d, st);
    return narrow ? launch_cfg<GemmCfg<MODE, 128, 4, false, H, H>, MODE>(d, st)
                  : launch_cfg<GemmCfg<MODE, 256, 4, false, H, H>, MODE>(d, st);
  }
  if constexpr (MODE == 0) {
    if (d.out_f32 && !d.aux_f32) return launch_cfg<GemmCfg<0, 256, 4, true, float, H>, 0>(d, st);
    if (d.out_f32 && d.aux_f32) return launch_cfg<GemmCfg<0, 256, 4, true, float, float>, 0>(d, st);
    if (!d.out_f32 && !d.aux_f32) return launch_cfg<GemmCfg<0, 256, 4, true, H, H>, 0>(d, st);
    set_error("gemm: bf16 output with fp32 aux is not instantiated");
    return MSMD_ERR_UNSUPPORTED;
  } else {
    set_error("gemm: the one-pass fp16 mode has no residual (aux) epilogue");
    return MSMD_ERR_UNSUPPORTED;
  }
}

int gemm_tc_launch(const GemmDesc& d, cudaStream_t st) {
  MSMD_REQUIRE(d.M > 0 && d.N > 0 && d.K > 0, "gemm: empty problem %dx%dx%d", d.M, d.N, d.K);
  MSMD_REQUIRE(d.A && d.W && d.out, "gemm: null operand");
  const bool aux = d.aux != nullptr;
  if (d.mode == 0) return dispatch16<0, __nv_bfloat16>(d, st);
  if (d.mode == 3) return dispatch16<3, __half>(d, st);
  MSMD_REQUIRE(d.mode == 1 || d.mode == 2, "gemm: unknown mode %d", d.mode);
  MSMD_REQUIRE(d.out_f32 && (!aux || d.aux_f32), "gemm: the three-pass modes are fp32 out");
  if (d.mode == 2) {
    if (aux) return launch_cfg<GemmCfg<2, 128, 4, true, float, float>, 2>(d, st);
    if (d.batch <= 1 && d.N >= 256 && d.M >= 2048)
      return launch_cfg<GemmCfg<2, 128, 4, false, float, float, true>, 2>(d, st);
    return launch_cfg<GemmCfg<2, 128, 4, false, float, float>, 2>(d, st);
  }
  if (aux) return launch_cfg<GemmCfg<1, 128, 4, true, float, float>, 1>(d, st);
  return launch_cfg<GemmCfg<1, 128, 4, false, float, float>, 1>(d, st);
}

// tf32 hi/lo split of an fp32 array (hi = value with the low 13 mantissa bits cleared, lo = value - hi)
__global__ void split_tf32_kernel(const float* __restrict__ x, float* __restrict__ hi, float* __restrict__ lo, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float v = x[i];
    const float h = __uint_as_float(__float_as_uint(v) & 0xffffe000u);
    hi[i] = h;
    lo[i] = v - h;
  }
}

// fp16 two-term split: hi = fp16(x), lo = fp16((x - hi) * 2^11); x ~= hi + 2^-11 lo to 22 mantissa bits
__global__ void split_f16_kernel(const float* __restrict__ x, __half* __restrict__ hi, __half* __restrict__ lo, int64_t n,
                                 int* __restrict__ overflow) {
  bool bad = false;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float v = x[i];
    const __half h = __float2half_rn(v);
    hi[i] = h;
    lo[i] = __float2half_rn((v - __half2float(h)) * 2048.0f);
    bad |= !(fabsf(v) <= 65504.0f);   // outside the fp16 range (or NaN): the split cannot represent it
  }
  if (bad && overflow) *overflow = 1;
}
int split_f16(const float* x, __half* hi, __half* lo, int64_t n, cudaStream_t st, int* overflow) {
  if (n == 0) return MSMD_OK;
  ProfileScope prof("split_f16", st);
  const int blocks = (int)std::min<int64_t>(cdiv(n, 256), kNumSMs * 16);
  split_f16_kernel<<<blocks, 256, 0, st>>>(x, hi, lo, n, overflow);
  MSMD_CHECK_LAUNCH();
  return MSMD_OK;
}

int split_tf32(const float* x, float* hi, float* lo, int64_t n, cudaStream_t st) {
  if (n == 0) return MSMD_OK;
  const int blocks = (int)std::min<int64_t>((n + 255) / 256, (int64_t)kNumSMs * 8);
  split_tf32_kernel<<<blocks, 256, 0, st>>>(x, hi, lo, n);
  MSMD_CHECK_LAUNCH();
  return MSMD_OK;
}

}  // namespace msmd

using namespace msmd;

// y = act(x W^T + b) (+ aux): the nn.Linear calls of model.py:931-961 / style_encoder.py / HF encoder.
extern "C" int msmd_linear(int mode, const void* x, const void* x_lo, const void* w, const void* w_lo,
                           const float* bias, const void* aux, void* out, int M, int N, int K, int64_t ldx,
                           int64_t ldw, int64_t ldo, int64_t ld_aux, int out_f32, int aux_f32, int act, void* stream) {
  GemmDesc d;
  d.mode = mode; d.A = x; d.A_lo = x_lo; d.W = w; d.W_lo = w_lo; d.bias = bias; d.aux = aux; d.out = out;
  d.M = M; d.N = N; d.K = K; d.lda = ldx; d.ldw = ldw; d.ldo = ldo; d.ld_aux = ld_aux;
  d.out_f32 = out_f32; d.aux_f32 = aux_f32; d.act = act & 1; d.gelu_heavy = (act & 1);
  return gemm_tc_launch(d, static_cast<cudaStream_t>(stream));
}

extern "C" int msmd_split_f16(const float* x, void* hi, void* lo, int64_t n, void* stream) {
  MSMD_REQUIRE(n >= 0, "msmd_split_f16: negative count");
  MSMD_REQUIRE(n == 0 || (x && hi && lo), "msmd_split_f16: null pointer");
  return split_f16(x, static_cast<__half*>(hi), static_cast<__half*>(lo), n, static_cast<cudaStream_t>(stream), nullptr);
}

extern "C" int msmd_split_tf32(const float* x, float* hi, float* lo, int64_t n, void* stream) {
  MSMD_REQUIRE(n >= 0, "msmd_split_tf32: negative count");
  MSMD_REQUIRE(n == 0 || (x && hi && lo), "msmd_split_tf32: null pointer");
  return split_tf32(x, hi, lo, n, static_cast<cudaStream_t>(stream));
}
