// Denoiser + sampler engine behind msmd_create / msmd_load_weights / msmd_window_begin / msmd_denoise /
// msmd_sample_window (include/msmd_b200.h).  Replaces model.py:820-996 and the loop at model.py:377-435.
//
// Data layout in HBM (S sequences, T = 1+Lp+L tokens, M = S*T rows, d = 512):
//   x     [M, d]     bf16   residual stream = A operand of every GEMM (token-major, features contiguous)
//   y     [M, d]     bf16   sub-layer outputs (out-proj / FF2 epilogues); the residual add happens in the LN kernel
//   qkv   [M, 3d]    bf16   packed q|k|v
//   ctx   [M, d]     bf16   attention output
//   h     [M, d_ff]  bf16   GELU(FF1)
//   kv[l] [S*(T-1), 2d] bf16 and ca[l] [S, T-1, d] bf16: per-window cross-attention caches (ca only at align_mask_width 1)
//   dec   [M, 80]    fp32   motion_dec output (67 dynamic + 4 alphas, row stride padded to 80)
#include "denoiser_kernels.cuh"
#include "gemm_tc.cuh"
#include "profile.cuh"
#include <cuda_fp16.h>
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <tuple>
#include <vector>

using namespace msmd;

namespace {

struct LayerW {
  bf16 *Wqkv = nullptr, *Wo = nullptr, *Wq0 = nullptr, *Wkv = nullptr, *Wco = nullptr, *W1 = nullptr, *W2 = nullptr;
  float *bqkv = nullptr, *bo = nullptr, *bq0 = nullptr, *bkv = nullptr, *bco = nullptr, *b1 = nullptr, *b2 = nullptr;
  float *g1 = nullptr, *be1 = nullptr, *g2 = nullptr, *be2 = nullptr, *g3 = nullptr, *be3 = nullptr;
  bf16 *kv = nullptr, *ca = nullptr;  // per-window caches (bf16 steps)
  bf16 *kvh = nullptr, *cah = nullptr;  // same in fp16 storage (one-pass fp16 steps)
  // fp32-grade path (precision >= 1): fp16 two-term splits (x = hi + 2^-11 lo, gemm_tc.cuh MODE 2) of the same
  // weights, and fp32 caches
  __half *Wqkv_h = nullptr, *Wqkv_l = nullptr, *Wo_h = nullptr, *Wo_l = nullptr, *Wq0_h = nullptr, *Wq0_l = nullptr,
         *Wkv_h = nullptr, *Wkv_l = nullptr, *Wco_h = nullptr, *Wco_l = nullptr, *W1_h = nullptr, *W1_l = nullptr,
         *W2_h = nullptr, *W2_l = nullptr;
  float *kv32 = nullptr, *ca32 = nullptr;
};

uint16_t f2bf(float f) {  // round-to-nearest-even
  uint32_t u;
  memcpy(&u, &f, 4);
  if ((u & 0x7fffffffu) > 0x7f800000u) return (uint16_t)((u >> 16) | 0x40);
  u += 0x7fffu + ((u >> 16) & 1u);
  return (uint16_t)(u >> 16);
}

}  // namespace

struct msmd_model {
  msmd_config c{};
  int device = 0;
  bool loaded = false, window = false;
  int T = 0, dp = 0, ldd = 80;
  std::vector<LayerW> L;
  std::vector<void*> owned;   // workspaces, freed in destroy
  std::vector<void*> wowned;  // packed weights: released and re-packed by every msmd_load_weights
  bool packing = false;       // dalloc target: wowned while load_weights runs
  // fp32 parameters
  float *PE = nullptr, *temb = nullptr, *Wp = nullptr, *bp = nullptr, *Wf = nullptr, *WfT = nullptr, *bf_ = nullptr;
  __half* Wf16 = nullptr;     // [2][d][80] fp16 hi | lo of feature_proj.weight[:, :dm] (tensor-core embedding)
  std::vector<float*> Ws0, bs0, Ws2, bs2;
  bf16 *Wd1 = nullptr, *Wd2 = nullptr;
  float *bd1 = nullptr, *bd2 = nullptr;
  float *alphas = nullptr, *alpha_bars = nullptr, *sig_flex = nullptr, *sig_inflex = nullptr;
  // workspaces
  bf16 *x = nullptr, *qkv = nullptr, *ctx = nullptr, *h = nullptr, *dec1 = nullptr, *mem = nullptr, *x0c = nullptr;
  bf16 *y = nullptr, *memh = nullptr;
  float *dec2 = nullptr, *pp = nullptr, *pmproj = nullptr, *stat = nullptr,
        *hid = nullptr, *xbuf = nullptr, *mixed = nullptr, *thr = nullptr;
  int* steps = nullptr;
  // fp32-grade path workspaces
  __half *Wd1_h = nullptr, *Wd1_l = nullptr, *Wd2_h = nullptr, *Wd2_l = nullptr;
  float *fx = nullptr, *fqkv = nullptr, *fctx = nullptr, *fh = nullptr, *fy = nullptr, *fdec1 = nullptr, *fmem = nullptr,
        *fx0c = nullptr, *fq0 = nullptr, *fctx0 = nullptr, *fy0 = nullptr;
  __half *ws_hi = nullptr, *ws_lo = nullptr;   // split scratch of the current A operand
  int* overflow = nullptr;                     // raised by the operand split when an activation leaves the fp16 range
  int *h_overflow = nullptr;                   // pinned mirror, filled asynchronously after fp32-grade steps
  cudaEvent_t ovf_event = nullptr;
  bool ovf_pending = false;
  bool window16[2] = {false, false}, window32 = false;   // per-window caches built for [bf16, fp16] / fp32-grade
  float *w_audio = nullptr, *w_prev_audio = nullptr, *w_ind = nullptr;   // engine-owned copies of the window's conditioning
  // window state
  int S = 0, NX = 0, E = 0;
  const float* indicator = nullptr;            // = w_ind, or null when the model has no indicator column
  // sampling loop: device-resident parameter block of the update kernel + instantiated step graphs, keyed by
  // (format, S, NX, E, thresholding).  Nothing caller-owned is baked into a graph, so it is reused by every later
  // window / call of the same shape; the capture stream is created once here.
  UpdateParams* d_up = nullptr;
  unsigned int* d_done = nullptr;   // block-completion counter of the update kernel
  long long* d_keys = nullptr;      // [max_seqs][2] per-clip Philox keys of the current call (msmd_sample_extras.noise_keys)
  SchedStep* d_sched = nullptr;     // [n_diff_steps + 1] respaced-step table of the current call, indexed by t
  float* d_hist = nullptr;          // [max_seqs, L, dm] data prediction of the last executed DPM-Solver++(2M) step, per row
  std::vector<double> h_alpha_bars; // host copy of diffusion_sched.alpha_bars: the respaced coefficients are planned on the host
  cudaStream_t cap_stream = nullptr;
  typedef std::tuple<int, int, int, int, int, float, float, float> GraphKey;
  std::map<GraphKey, cudaGraphExec_t> graphs;
  void drop_graphs() {
    for (auto& g : graphs) cudaGraphExecDestroy(g.second);
    graphs.clear();
  }
};

namespace {

template <class Tp>
int dalloc(msmd_model* m, Tp** p, size_t n) {
  void* q = nullptr;
  MSMD_CHECK_CUDA(cudaMalloc(&q, n * sizeof(Tp)));
  (m->packing ? m->wowned : m->owned).push_back(q);
  *p = static_cast<Tp*>(q);
  return MSMD_OK;
}

int up_f32(msmd_model* m, float** dst, const std::vector<float>& h) {
  int rc = dalloc(m, dst, h.size());
  if (rc) return rc;
  MSMD_CHECK_CUDA(cudaMemcpy(*dst, h.data(), h.size() * 4, cudaMemcpyHostToDevice));
  return MSMD_OK;
}
int up_bf16(msmd_model* m, bf16** dst, const float* h, size_t n) {
  std::vector<uint16_t> t(n);
  for (size_t i = 0; i < n; ++i) t[i] = f2bf(h[i]);
  int rc = dalloc(m, dst, n);
  if (rc) return rc;
  MSMD_CHECK_CUDA(cudaMemcpy(*dst, t.data(), n * 2, cudaMemcpyHostToDevice));
  return MSMD_OK;
}

// one-pass 16-bit GEMM: fmt 0 = bf16 operands (gemm_tc MODE 0), 1 = fp16 operands (MODE 3); W is the matching copy
int gemm(int fmt, const bf16* A, int64_t lda, const void* W, int64_t ldw, const float* bias, const bf16* aux, int64_t ld_aux,
         void* out, int64_t ldo, int out_f32, int M, int N, int K, int act, cudaStream_t st) {
  GemmDesc d;
  d.mode = fmt ? 3 : 0; d.A = A; d.W = W; d.bias = bias; d.aux = aux; d.out = out;
  d.M = M; d.N = N; d.K = K; d.lda = lda; d.ldw = ldw; d.ldo = ldo; d.ld_aux = ld_aux;
  d.out_f32 = out_f32; d.aux_f32 = 0; d.act = act; d.gelu_heavy = act;
  return gemm_tc_launch(d, st);
}

// fp16 copies of a weight: hi = fp16(w) (also the operand of the one-pass fp16 steps) and, for the fp32-grade path,
// lo = fp16((w - hi) * 2^11)
int up_split(msmd_model* m, __half** hi, __half** lo, const float* h, size_t n, bool want_lo) {
  std::vector<__half> a(n), b(want_lo ? n : 0);
  for (size_t i = 0; i < n; ++i) {
    a[i] = __float2half_rn(h[i]);
    if (want_lo) b[i] = __float2half_rn((h[i] - __half2float(a[i])) * 2048.0f);
  }
  int rc;
  if ((rc = dalloc(m, hi, n))) return rc;
  MSMD_CHECK_CUDA(cudaMemcpy(*hi, a.data(), n * sizeof(__half), cudaMemcpyHostToDevice));
  if (want_lo) {
    if ((rc = dalloc(m, lo, n))) return rc;
    MSMD_CHECK_CUDA(cudaMemcpy(*lo, b.data(), n * sizeof(__half), cudaMemcpyHostToDevice));
  }
  return MSMD_OK;
}

// fp32-grade linear: split the activations (fp16 hi + scaled fp16 residual), then the 3-pass tcgen05 GEMM
int gemm32(msmd_model* m, const float* A, int64_t lda, const __half* Wh, const __half* Wl, int64_t ldw, const float* bias,
           float* out, int64_t ldo, int M, int N, int K, int act, cudaStream_t st) {
  int rc;
  // the split kernel works on contiguous [M, lda] storage; K <= lda columns are used by the GEMM
  if ((rc = split_f16(A, m->ws_hi, m->ws_lo, (int64_t)(M - 1) * lda + K, st, m->overflow))) return rc;
  GemmDesc d;
  d.mode = 2; d.A = m->ws_hi; d.A_lo = m->ws_lo; d.W = Wh; d.W_lo = Wl; d.bias = bias; d.out = out;
  d.M = M; d.N = N; d.K = K; d.lda = lda; d.ldw = ldw; d.ldo = ldo; d.out_f32 = 1; d.aux_f32 = 1; d.act = act;
  return gemm_tc_launch(d, st);
}

int window_begin_f32(msmd_model* m, cudaStream_t st);

// fp32-grade forward (same graph of operations as run_forward, fp32 activations, tf32x3 GEMMs)
int run_forward_f32(msmd_model* m, const float* xrows, cudaStream_t st) {
  const msmd_config& c = m->c;
  const int S = m->S, T = m->T, d = c.d_model, M = S * T;
  int rc;
  if (!m->window32 && (rc = window_begin_f32(m, st))) return rc;
  EmbedParams ep{};
  ep.pp = m->pp; ep.temb = m->temb; ep.pmproj = m->pmproj; ep.PE = m->PE; ep.steps = m->steps;
  ep.x = xrows; ep.indicator = c.use_indicator ? m->indicator : nullptr; ep.WfT = m->WfT; ep.bf = m->bf_;
  ep.out = nullptr; ep.S = S; ep.NX = m->NX; ep.E = m->E; ep.Lp = c.n_prev_motions; ep.L = c.n_motions; ep.d = d;
  ep.dm = c.motion_dim;
  if ((rc = embed_f32_launch(ep, m->fx, st))) return rc;
  for (int l = 0; l < c.n_layers; ++l) {
    LayerW& w = m->L[l];
    if ((rc = gemm32(m, m->fx, d, w.Wqkv_h, w.Wqkv_l, d, w.bqkv, m->fqkv, 3 * d, M, 3 * d, d, 0, st))) return rc;
    if ((rc = self_attn_f32_launch(m->fqkv, m->fctx, S, T, c.n_heads, st))) return rc;
    if ((rc = gemm32(m, m->fctx, d, w.Wo_h, w.Wo_l, d, w.bo, m->fy, d, M, d, d, 0, st))) return rc;
    if (c.align_mask_width == 1) {
      if ((rc = ln_f32_launch(m->fy, m->fx, w.g1, w.be1, w.ca32, w.g2, w.be2, m->fx, m->fx0c, M, T, st))) return rc;
      if ((rc = gemm32(m, m->fx0c, d, w.Wq0_h, w.Wq0_l, d, w.bq0, m->fq0, d, S, d, d, 0, st))) return rc;
      if ((rc = cross_attn_row0_f32_launch(m->fq0, w.kv32, m->fctx0, S, T - 1, c.n_heads, st))) return rc;
      if ((rc = gemm32(m, m->fctx0, d, w.Wco_h, w.Wco_l, d, w.bco, m->fy0, d, S, d, d, 0, st))) return rc;
      if ((rc = ln_row0_f32_launch(m->fy0, m->fx0c, w.g2, w.be2, m->fx, S, T, st))) return rc;
    } else {   // banded cross attention of every row (q into the free qkv workspace), out-proj, residual + norm2
      if ((rc = ln_f32_launch(m->fy, m->fx, w.g1, w.be1, nullptr, nullptr, nullptr, m->fx, nullptr, M, T, st))) return rc;
      if ((rc = gemm32(m, m->fx, d, w.Wq0_h, w.Wq0_l, d, w.bq0, m->fqkv, d, M, d, d, 0, st))) return rc;
      if ((rc = cross_attn_f32_launch(m->fqkv, w.kv32, m->fctx, S, T, T - 1, c.n_heads, c.align_mask_width, st))) return rc;
      if ((rc = gemm32(m, m->fctx, d, w.Wco_h, w.Wco_l, d, w.bco, m->fy, d, M, d, d, 0, st))) return rc;
      if ((rc = ln_f32_launch(m->fy, m->fx, w.g2, w.be2, nullptr, nullptr, nullptr, m->fx, nullptr, M, T, st))) return rc;
    }
    if ((rc = gemm32(m, m->fx, d, w.W1_h, w.W1_l, d, w.b1, m->fh, c.d_ff, M, c.d_ff, d, 1, st))) return rc;
    if ((rc = gemm32(m, m->fh, c.d_ff, w.W2_h, w.W2_l, c.d_ff, w.b2, m->fy, d, M, d, c.d_ff, 0, st))) return rc;
    if ((rc = ln_f32_launch(m->fy, m->fx, w.g3, w.be3, nullptr, nullptr, nullptr, m->fx, nullptr, M, T, st))) return rc;
  }
  if ((rc = gemm32(m, m->fx, d, m->Wd1_h, m->Wd1_l, d, m->bd1, m->fdec1, d / 2, M, d / 2, d, 1, st))) return rc;
  if ((rc = gemm32(m, m->fdec1, d / 2, m->Wd2_h, m->Wd2_l, d / 2, m->bd2, m->dec2, m->ldd, M, c.motion_dim + c.n_basis,
                   d / 2, 0, st)))
    return rc;
  return MSMD_OK;
}

// per-window caches of the fp32-grade path (built lazily: the hybrid schedule only needs them for its last steps)
int window_begin_f32(msmd_model* m, cudaStream_t st) {
  const msmd_config& c = m->c;
  const int S = m->S, d = c.d_model, Tk = m->T - 1;
  int rc;
  if ((rc = build_memory_f32(m->w_prev_audio, m->w_audio, m->fmem, S, c.n_prev_motions, c.n_motions, d, st))) return rc;
  for (auto& w : m->L) {
    if ((rc = gemm32(m, m->fmem, d, w.Wkv_h, w.Wkv_l, d, w.bkv, w.kv32, 2 * d, S * Tk, 2 * d, d, 0, st))) return rc;
    if (c.align_mask_width != 1) continue;   // the motion rows' attention depends on the query: no ca cache
    // v half of the kv cache as a strided A operand: row stride 2d, K = d columns starting at column d
    if ((rc = split_f16(w.kv32, m->ws_hi, m->ws_lo, (int64_t)S * Tk * 2 * d, st, m->overflow))) return rc;
    GemmDesc g;
    g.mode = 2; g.A = m->ws_hi + d; g.A_lo = m->ws_lo + d; g.W = w.Wco_h; g.W_lo = w.Wco_l; g.bias = w.bco; g.out = w.ca32;
    g.M = S * Tk; g.N = d; g.K = d; g.lda = 2 * d; g.ldw = d; g.ldo = d; g.out_f32 = 1; g.aux_f32 = 1;
    if ((rc = gemm_tc_launch(g, st))) return rc;
  }
  m->window32 = true;
  return MSMD_OK;
}

// One forward of the network on the current window context: x rows [NX,L,dm] -> dec2 [M, ldd].
// fmt 0: bf16 storage + bf16 tensor-core GEMMs; fmt 1: fp16 storage + one-pass fp16 GEMMs (same kernels, same cost,
// 11 mantissa bits instead of 8: x0_hat error 8e-4 instead of 6.5e-3).
int run_forward(msmd_model* m, const float* xrows, cudaStream_t st, int fmt) {
  const msmd_config& c = m->c;
  const int S = m->S, T = m->T, d = c.d_model, M = S * T;
  int rc;
  EmbedParams ep{};
  ep.pp = m->pp; ep.temb = m->temb; ep.pmproj = m->pmproj; ep.PE = m->PE; ep.steps = m->steps;
  ep.x = xrows; ep.indicator = c.use_indicator ? m->indicator : nullptr; ep.WfT = m->WfT; ep.bf = m->bf_;
  ep.out = m->x; ep.S = S; ep.NX = m->NX; ep.E = m->E; ep.Lp = c.n_prev_motions; ep.L = c.n_motions; ep.d = d;
  ep.dm = c.motion_dim; ep.fp16 = fmt; ep.Wf16 = m->Wf16;
  if ((rc = embed_launch(ep, st))) return rc;
  for (int l = 0; l < c.n_layers; ++l) {
    LayerW& w = m->L[l];
    const void *Wqkv = fmt ? (const void*)w.Wqkv_h : w.Wqkv, *Wo = fmt ? (const void*)w.Wo_h : w.Wo,
               *Wq0 = fmt ? (const void*)w.Wq0_h : w.Wq0, *Wco = fmt ? (const void*)w.Wco_h : w.Wco,
               *W1 = fmt ? (const void*)w.W1_h : w.W1, *W2 = fmt ? (const void*)w.W2_h : w.W2;
    const bf16 *kv = fmt ? w.kvh : w.kv, *ca = fmt ? w.cah : w.ca;
    // self-attention block (nn.TransformerDecoderLayer._sa_block) + norm1, then (width 1) the cached cross-attention
    // rows + norm2 for motion tokens
    if ((rc = gemm(fmt, m->x, d, Wqkv, d, w.bqkv, nullptr, 0, m->qkv, 3 * d, 0, M, 3 * d, d, 0, st))) return rc;
    if ((rc = self_attn_tc_launch(m->qkv, m->ctx, S, T, c.n_heads, fmt, st))) return rc;
    if ((rc = gemm(fmt, m->ctx, d, Wo, d, w.bo, nullptr, 0, m->y, d, 0, M, d, d, 0, st))) return rc;
    LnParams lp{};
    lp.resid = m->x;
    lp.y = m->y; lp.g1 = w.g1; lp.b1 = w.be1; lp.add = ca; lp.g2 = w.g2; lp.b2 = w.be2; lp.out = m->x;
    lp.x0 = m->x0c; lp.M = M; lp.T = T; lp.d = d; lp.fp16 = fmt;
    if (c.align_mask_width != 1) {
      // banded cross attention (_mha_block with the alignment mask) of every row, person token included, on every step:
      // norm1 of all rows, q projection into the qkv workspace (free after self-attention), attention over the cached
      // K|V, out-proj, then residual + norm2
      lp.add = nullptr; lp.g2 = nullptr; lp.b2 = nullptr; lp.x0 = nullptr;
      if ((rc = ln_launch(lp, st))) return rc;
      if ((rc = gemm(fmt, m->x, d, Wq0, d, w.bq0, nullptr, 0, m->qkv, d, 0, M, d, d, 0, st))) return rc;
      if ((rc = cross_attn_tc_launch(m->qkv, kv, m->ctx, S, T, T - 1, c.n_heads, c.align_mask_width, fmt, st))) return rc;
      if ((rc = gemm(fmt, m->ctx, d, Wco, d, w.bco, nullptr, 0, m->y, d, 0, M, d, d, 0, st))) return rc;
      LnParams l2 = lp;
      l2.g1 = w.g2; l2.b1 = w.be2;
      if ((rc = ln_launch(l2, st))) return rc;
    } else {
      if ((rc = ln_launch(lp, st))) return rc;
      // person token (row 0): real cross attention over the memory (_mha_block) + norm2 as one cluster kernel
      // (row0_fused.cu)
      if ((rc = row0_fused_launch(m->x0c, static_cast<const bf16*>(Wq0), w.bq0, kv, static_cast<const bf16*>(Wco), w.bco,
                                  w.g2, w.be2, m->x, S, T, T - 1, c.n_heads, d, fmt, st)))
        return rc;
    }
    // feed-forward block (_ff_block) + norm3
    if ((rc = gemm(fmt, m->x, d, W1, d, w.b1, nullptr, 0, m->h, c.d_ff, 0, M, c.d_ff, d, 1, st))) return rc;
    if ((rc = gemm(fmt, m->h, c.d_ff, W2, c.d_ff, w.b2, nullptr, 0, m->y, d, 0, M, d, c.d_ff, 0, st))) return rc;
    LnParams l3{};
    l3.resid = m->x;
    l3.y = m->y; l3.g1 = w.g3; l3.b1 = w.be3; l3.add = nullptr; l3.g2 = nullptr; l3.b2 = nullptr; l3.out = m->x;
    l3.x0 = nullptr; l3.M = M; l3.T = T; l3.d = d; l3.fp16 = fmt;
    if ((rc = ln_launch(l3, st))) return rc;
  }
  // motion_dec (model.py:961): Linear(d, d/2) + GELU + Linear(d/2, dm + n_basis)
  const void *Wd1 = fmt ? (const void*)m->Wd1_h : m->Wd1, *Wd2 = fmt ? (const void*)m->Wd2_h : m->Wd2;
  if ((rc = gemm(fmt, m->x, d, Wd1, d, m->bd1, nullptr, 0, m->dec1, d / 2, 0, M, d / 2, d, 1, st))) return rc;
  if ((rc = gemm(fmt, m->dec1, d / 2, Wd2, d / 2, m->bd2, nullptr, 0, m->dec2, m->ldd, 1, M, c.motion_dim + c.n_basis,
                 d / 2, 0, st)))
    return rc;
  return MSMD_OK;
}

// per-window caches of a 16-bit path (fmt 0 bf16 / 1 fp16): memory K|V projection of every layer, then, at
// align_mask_width 1, the motion rows' cross-attention output out_proj(v_proj(mem)) (softmax over a single visible key
// is 1, so the query drops out: SURVEY section 0).  Built on first use in the window: a pure-bf16 call never pays for
// the fp16 copies.
int window_begin_16(msmd_model* m, int fmt, cudaStream_t st) {
  const msmd_config& c = m->c;
  const int S = m->S, d = c.d_model, Tk = m->T - 1;
  int rc;
  bf16* mem = fmt ? m->memh : m->mem;
  if ((rc = build_memory_h16(m->w_prev_audio, m->w_audio, mem, S, c.n_prev_motions, c.n_motions, d, fmt, st))) return rc;
  for (auto& w : m->L) {
    bf16 *kv = fmt ? w.kvh : w.kv, *ca = fmt ? w.cah : w.ca;
    const void *Wkv = fmt ? (const void*)w.Wkv_h : w.Wkv, *Wco = fmt ? (const void*)w.Wco_h : w.Wco;
    if ((rc = gemm(fmt, mem, d, Wkv, d, w.bkv, nullptr, 0, kv, 2 * d, 0, S * Tk, 2 * d, d, 0, st))) return rc;
    if (c.align_mask_width == 1 && (rc = gemm(fmt, kv + d, 2 * d, Wco, d, w.bco, nullptr, 0, ca, d, 0, S * Tk, d, d, 0, st)))
      return rc;
  }
  m->window16[fmt] = true;
  return MSMD_OK;
}

// which arithmetic a model created with `precision` holds
bool has_bf16(const msmd_config& c) { return c.precision == 0 || c.precision == 2; }
bool has_fp16(const msmd_config& c) { return c.precision == 2 || c.precision == 3; }
bool has_f32(const msmd_config& c) { return c.precision == 1 || c.precision == 2; }

// The fp32-grade path reports operand-split overflow without synchronising the call that hit it: the flag is copied
// to pinned memory behind the work, and inspected here at the NEXT entry (the state itself was poisoned with NaN).
int poll_overflow(msmd_model* m, const char* who) {
  if (!m->ovf_pending || cudaEventQuery(m->ovf_event) != cudaSuccess) return MSMD_OK;
  m->ovf_pending = false;
  if (*m->h_overflow) {
    *m->h_overflow = 0;
    cudaMemset(m->overflow, 0, sizeof(int));
    set_error("%s: an earlier fp32-grade call left the fp16 range of its GEMM operand split (|activation| > 65504 or NaN); "
              "its output was poisoned with NaN", who);
    return MSMD_ERR_INVALID;
  }
  return MSMD_OK;
}
int post_overflow(msmd_model* m, cudaStream_t st) {
  MSMD_CHECK_CUDA(cudaMemcpyAsync(m->h_overflow, m->overflow, sizeof(int), cudaMemcpyDeviceToHost, st));
  MSMD_CHECK_CUDA(cudaEventRecord(m->ovf_event, st));
  m->ovf_pending = true;
  return MSMD_OK;
}

}  // namespace

extern "C" int msmd_create(const msmd_config* cfg, int device, msmd_model** out) {
  MSMD_REQUIRE(cfg && out, "msmd_create: null argument");
  const msmd_config& c = *cfg;
  // supported shape envelope (ADVICE r1): the kernels are specialised for the released architecture
  MSMD_REQUIRE(c.d_model == 512 && c.n_heads * 64 == c.d_model, "msmd_create: only d_model=512 / 8 heads x 64 is built (got %d / %d)",
               c.d_model, c.n_heads);
  MSMD_REQUIRE(c.n_motions > 0 && c.n_prev_motions >= 0 && 1 + c.n_prev_motions + c.n_motions <= 112,
               "msmd_create: sequence 1 + n_prev_motions + n_motions = %d exceeds the 112-token attention tile "
               "(the released configuration is 1 + 10 + 100)", 1 + c.n_prev_motions + c.n_motions);
  MSMD_REQUIRE(c.n_layers > 0 && c.d_ff > 0 && c.d_ff % 8 == 0 && c.max_seqs > 0 && c.n_diff_steps > 0, "msmd_create: bad sizes");
  MSMD_REQUIRE(c.n_basis >= 1, "msmd_create: n_basis=%d (the network mixes its output from at least one static basis: "
               "the reference cannot run num_of_basis = 0)", c.n_basis);
  MSMD_REQUIRE(c.motion_dim > 3 && c.motion_dim + c.n_basis <= 80, "msmd_create: motion_dim + n_basis > 80");
  MSMD_REQUIRE(c.align_mask_width >= 0, "msmd_create: align_mask_width=%d (0 = no alignment mask, w >= 1 = band of 2w-1 "
               "memory tokens)", c.align_mask_width);
  MSMD_REQUIRE(c.precision >= 0 && c.precision <= 3,
               "msmd_create: precision %d (0 bf16, 1 fp32-grade, 2 hybrid: bf16 + fp16 + fp32-grade, 3 fp16)", c.precision);
  MSMD_CHECK_CUDA(cudaSetDevice(device));
  msmd_model* m = new msmd_model();
  m->c = c;
  m->device = device;
  m->T = 1 + c.n_prev_motions + c.n_motions;
  m->dp = c.d_shape + c.d_style;
  m->L.resize(c.n_layers);
  const size_t S = c.max_seqs, T = m->T, M = S * T, d = c.d_model;
  int rc = MSMD_OK;
  auto A = [&](auto** p, size_t n) { if (!rc) rc = dalloc(m, p, n); };
  A(&m->dec2, M * m->ldd); A(&m->pp, S * d);
  A(&m->pmproj, S * c.n_prev_motions * d); A(&m->stat, S * c.n_basis * c.motion_dim); A(&m->hid, S * d);
  A(&m->thr, S);
  A(&m->xbuf, S * c.n_motions * c.motion_dim); A(&m->mixed, S * (T - 1) * c.motion_dim); A(&m->steps, S);
  A(&m->w_audio, S * c.n_motions * d); A(&m->w_prev_audio, S * c.n_prev_motions * d); A(&m->w_ind, S * c.n_motions);
  A(&m->d_up, 1); A(&m->d_done, 1); A(&m->d_keys, S * 2); A(&m->d_sched, (size_t)c.n_diff_steps + 1);
  A(&m->d_hist, S * c.n_motions * c.motion_dim);
  if (has_bf16(c) || has_fp16(c)) {
    A(&m->x, M * d); A(&m->qkv, M * 3 * d); A(&m->ctx, M * d); A(&m->h, M * c.d_ff); A(&m->dec1, M * d / 2);
    A(&m->x0c, S * d); A(&m->y, M * d);
  }
  // the step-invariant cross-attention rows (ca / cah / ca32) exist only at align_mask_width 1
  const bool want_ca = c.align_mask_width == 1;
  if (has_bf16(c)) {
    A(&m->mem, S * (T - 1) * d);
    for (auto& w : m->L) { A(&w.kv, S * (T - 1) * 2 * d); if (want_ca) A(&w.ca, S * (T - 1) * d); }
  }
  if (has_fp16(c)) {
    A(&m->memh, S * (T - 1) * d);
    for (auto& w : m->L) { A(&w.kvh, S * (T - 1) * 2 * d); if (want_ca) A(&w.cah, S * (T - 1) * d); }
  }
  if (has_f32(c)) {
    A(&m->fx, M * d); A(&m->fqkv, M * 3 * d); A(&m->fctx, M * d); A(&m->fh, M * c.d_ff); A(&m->fy, M * d);
    A(&m->fdec1, M * d / 2); A(&m->fmem, S * (T - 1) * d); A(&m->fx0c, S * d); A(&m->fq0, S * d); A(&m->fctx0, S * d);
    A(&m->fy0, S * d);
    // split scratch of the current A operand: the widest is FF2's [M, d_ff] or the window pass's kv cache [S*Tk, 2d]
    const size_t ws = std::max(M * (size_t)c.d_ff, S * (T - 1) * 2 * d);
    A(&m->ws_hi, ws); A(&m->ws_lo, ws); A(&m->overflow, 1);
    for (auto& w : m->L) { A(&w.kv32, S * (T - 1) * 2 * d); if (want_ca) A(&w.ca32, S * (T - 1) * d); }
  }
  if (!rc && cudaStreamCreateWithFlags(&m->cap_stream, cudaStreamNonBlocking) != cudaSuccess) rc = MSMD_ERR_CUDA;
  if (!rc && m->overflow) {
    if (cudaMallocHost(&m->h_overflow, sizeof(int)) != cudaSuccess ||
        cudaEventCreateWithFlags(&m->ovf_event, cudaEventDisableTiming) != cudaSuccess)
      rc = MSMD_ERR_CUDA;
    else
      *m->h_overflow = 0;
  }
  if (rc) { msmd_destroy(m); return rc; }
  cudaMemset(m->dec2, 0, M * m->ldd * sizeof(float));
  cudaMemset(m->d_done, 0, sizeof(unsigned int));
  if (m->overflow) cudaMemset(m->overflow, 0, sizeof(int));
  *out = m;
  return MSMD_OK;
}

extern "C" void msmd_destroy(msmd_model* m) {
  if (!m) return;
  cudaSetDevice(m->device);
  cudaDeviceSynchronize();   // graph launches / async copies of earlier calls may still be in flight
  m->drop_graphs();
  if (m->cap_stream) cudaStreamDestroy(m->cap_stream);
  if (m->ovf_event) cudaEventDestroy(m->ovf_event);
  if (m->h_overflow) cudaFreeHost(m->h_overflow);
  for (void* p : m->owned) cudaFree(p);
  for (void* p : m->wowned) cudaFree(p);
  delete m;
}

extern "C" int msmd_load_weights(msmd_model* m, const char* const* names, const void* const* data,
                                 const int64_t* numel, int n) {
  MSMD_REQUIRE(m && names && data && numel, "msmd_load_weights: null argument");
  const msmd_config& c = m->c;
  MSMD_CHECK_CUDA(cudaSetDevice(m->device));
  // a reload replaces the previous packed copies (they used to accumulate until msmd_destroy) and invalidates the
  // step graphs, which hold their addresses
  MSMD_CHECK_CUDA(cudaDeviceSynchronize());
  m->drop_graphs();
  for (void* p : m->wowned) cudaFree(p);
  m->wowned.clear();
  m->loaded = false;
  m->window = false;
  struct PackScope { msmd_model* m; PackScope(msmd_model* mm) : m(mm) { m->packing = true; } ~PackScope() { m->packing = false; } } scope(m);
  std::map<std::string, int> idx;
  for (int i = 0; i < n; ++i) idx[names[i]] = i;
  std::string missing;
  int rc = MSMD_OK;
  auto fetch = [&](const std::string& key, size_t expect, std::vector<float>& h) -> bool {
    auto it = idx.find(key);
    if (it == idx.end()) { missing += key + " "; return false; }
    if ((size_t)numel[it->second] != expect) {
      set_error("msmd_load_weights: %s has %lld elements, expected %zu", key.c_str(), (long long)numel[it->second], expect);
      rc = MSMD_ERR_INVALID;
      return false;
    }
    h.resize(expect);
    if (cudaMemcpy(h.data(), data[it->second], expect * 4, cudaMemcpyDefault) != cudaSuccess) {
      set_error("msmd_load_weights: copy of %s failed", key.c_str());
      rc = MSMD_ERR_CUDA;
      return false;
    }
    return true;
  };
  const size_t d = c.d_model, ff = c.d_ff, dm = c.motion_dim, fin = dm + (c.use_indicator ? 1 : 0);
  const std::string P = "denoising_net.";
  std::vector<float> h, h2;
  auto F32 = [&](const std::string& key, size_t n_, float** dst) { if (!rc && fetch(key, n_, h)) rc = up_f32(m, dst, h); };
  const bool want_bf = has_bf16(c), want_hi = has_fp16(c) || has_f32(c), want_lo = has_f32(c);
  // a GEMM weight: bf16 copy for the bf16 path and/or fp16 hi (+ lo) for the one-pass fp16 / fp32-grade paths
  auto put_w = [&](const float* src, size_t n_, bf16** dst, __half** hi, __half** lo) {
    if (!rc && want_bf) rc = up_bf16(m, dst, src, n_);
    if (!rc && want_hi) rc = up_split(m, hi, lo, src, n_, want_lo);
  };
  auto BF = [&](const std::string& key, size_t n_, bf16** dst, __half** hi, __half** lo) {
    if (!rc && fetch(key, n_, h)) put_w(h.data(), n_, dst, hi, lo);
  };

  for (int l = 0; l < c.n_layers && !rc; ++l) {
    LayerW& w = m->L[l];
    const std::string q = P + "transformer.layers." + std::to_string(l) + ".";
    BF(q + "self_attn.in_proj_weight", 3 * d * d, &w.Wqkv, &w.Wqkv_h, &w.Wqkv_l);
    F32(q + "self_attn.in_proj_bias", 3 * d, &w.bqkv);
    BF(q + "self_attn.out_proj.weight", d * d, &w.Wo, &w.Wo_h, &w.Wo_l);
    F32(q + "self_attn.out_proj.bias", d, &w.bo);
    if (!rc && fetch(q + "multihead_attn.in_proj_weight", 3 * d * d, h)) {  // packed q|k|v (model.py:874 / App. E)
      put_w(h.data(), d * d, &w.Wq0, &w.Wq0_h, &w.Wq0_l);
      put_w(h.data() + d * d, 2 * d * d, &w.Wkv, &w.Wkv_h, &w.Wkv_l);
    }
    if (!rc && fetch(q + "multihead_attn.in_proj_bias", 3 * d, h)) {
      rc = up_f32(m, &w.bq0, std::vector<float>(h.begin(), h.begin() + d));
      if (!rc) rc = up_f32(m, &w.bkv, std::vector<float>(h.begin() + d, h.end()));
    }
    BF(q + "multihead_attn.out_proj.weight", d * d, &w.Wco, &w.Wco_h, &w.Wco_l);
    F32(q + "multihead_attn.out_proj.bias", d, &w.bco);
    BF(q + "linear1.weight", ff * d, &w.W1, &w.W1_h, &w.W1_l);
    F32(q + "linear1.bias", ff, &w.b1);
    BF(q + "linear2.weight", d * ff, &w.W2, &w.W2_h, &w.W2_l);
    F32(q + "linear2.bias", d, &w.b2);
    F32(q + "norm1.weight", d, &w.g1); F32(q + "norm1.bias", d, &w.be1);
    F32(q + "norm2.weight", d, &w.g2); F32(q + "norm2.bias", d, &w.be2);
    F32(q + "norm3.weight", d, &w.g3); F32(q + "norm3.bias", d, &w.be3);
  }
  F32(P + "PE", (size_t)m->T * d, &m->PE);
  F32(P + "person_proj.weight", d * m->dp, &m->Wp);
  F32(P + "person_proj.bias", d, &m->bp);
  if (!rc && fetch(P + "feature_proj.weight", d * fin, h)) {
    rc = up_f32(m, &m->Wf, h);
    std::vector<float> t((dm + 1) * d, 0.f);  // k-major copy; row dm = indicator column (zero if unused)
    for (size_t cc = 0; cc < d; ++cc)
      for (size_t k = 0; k < fin; ++k) t[k * d + cc] = h[cc * fin + k];
    if (!rc) rc = up_f32(m, &m->WfT, t);
    if (!rc) {   // fp16 two-term split of the motion columns, [n][k] with K zero-padded to 80 (embed_x_mma_kernel)
      std::vector<__half> w16(2 * d * 80, __float2half_rn(0.f));
      for (size_t cc = 0; cc < d; ++cc)
        for (size_t k = 0; k < dm; ++k) {
          const float v = h[cc * fin + k];
          const __half hi = __float2half_rn(v);
          w16[cc * 80 + k] = hi;
          w16[d * 80 + cc * 80 + k] = __float2half_rn(v - __half2float(hi));
        }
      rc = dalloc(m, &m->Wf16, w16.size());
      if (!rc) MSMD_CHECK_CUDA(cudaMemcpy(m->Wf16, w16.data(), w16.size() * sizeof(__half), cudaMemcpyHostToDevice));
    }
  }
  F32(P + "feature_proj.bias", d, &m->bf_);
  m->Ws0.assign(c.n_basis, nullptr); m->bs0 = m->Ws2 = m->bs2 = m->Ws0;
  for (int b = 0; b < c.n_basis && !rc; ++b) {
    const std::string q = P + "static_feature_mapping." + std::to_string(b) + ".";
    F32(q + "0.weight", d * c.d_style, &m->Ws0[b]); F32(q + "0.bias", d, &m->bs0[b]);
    F32(q + "2.weight", dm * d, &m->Ws2[b]); F32(q + "2.bias", dm, &m->bs2[b]);
  }
  BF(P + "motion_dec.0.weight", (d / 2) * d, &m->Wd1, &m->Wd1_h, &m->Wd1_l);
  F32(P + "motion_dec.0.bias", d / 2, &m->bd1);
  BF(P + "motion_dec.2.weight", (dm + c.n_basis) * (d / 2), &m->Wd2, &m->Wd2_h, &m->Wd2_l);
  if (!rc && fetch(P + "motion_dec.2.bias", dm + c.n_basis, h)) {
    h.resize(m->ldd, 0.f);
    rc = up_f32(m, &m->bd2, h);
  }
  // timestep-embedding table: diff_step_map(TE.pe[0, t]) for t = 0..T (model.py:931) — weights only
  const size_t nt = c.n_diff_steps + 1;
  float *te = nullptr, *w0 = nullptr, *b0 = nullptr, *w2 = nullptr, *b2 = nullptr, *hid = nullptr;
  F32(P + "TE.pe", nt * d, &te);
  F32(P + "diff_step_map.0.weight", d * d, &w0); F32(P + "diff_step_map.0.bias", d, &b0);
  F32(P + "diff_step_map.2.weight", d * d, &w2); F32(P + "diff_step_map.2.bias", d, &b2);
  // schedule (model.py:20-71): copied, not recomputed (SURVEY 8(a) a6)
  F32("diffusion_sched.alphas", nt, &m->alphas);
  if (!rc && fetch("diffusion_sched.alpha_bars", nt, h)) {
    rc = up_f32(m, &m->alpha_bars, h);
    m->h_alpha_bars.assign(h.begin(), h.end());
  }
  F32("diffusion_sched.sigmas_flex", nt, &m->sig_flex);
  F32("diffusion_sched.sigmas_inflex", nt, &m->sig_inflex);
  if (rc) return rc;
  if (!missing.empty()) {
    set_error("msmd_load_weights: missing state_dict keys: %s", missing.c_str());
    return MSMD_ERR_INVALID;
  }
  if ((rc = dalloc(m, &hid, nt * d)) || (rc = dalloc(m, &m->temb, nt * d))) return rc;
  if ((rc = linear_simt(te, d, w0, d, b0, hid, d, (int)nt, (int)d, (int)d, 1, 0))) return rc;
  if ((rc = linear_simt(hid, d, w2, d, b2, m->temb, d, (int)nt, (int)d, (int)d, 0, 0))) return rc;
  MSMD_CHECK_CUDA(cudaDeviceSynchronize());
  m->loaded = true;
  return MSMD_OK;
}

extern "C" int msmd_window_begin(msmd_model* m, const float* audio, const float* person, const float* style,
                                 const float* prev_motion, const float* prev_audio, const float* indicator, int S,
                                 int NX, int E, void* stream) {
  MSMD_REQUIRE(m, "msmd_window_begin: null model");
  if (!m->loaded) { set_error("msmd_window_begin: weights not loaded"); return MSMD_ERR_STATE; }
  const msmd_config& c = m->c;
  MSMD_REQUIRE(S > 0 && NX > 0 && E > 0 && S == NX * E, "msmd_window_begin: S=%d must equal NX*E=%d*%d", S, NX, E);
  MSMD_REQUIRE(S <= c.max_seqs, "msmd_window_begin: %d sequences exceed the capacity %d given at create", S, c.max_seqs);
  MSMD_REQUIRE(E <= 3, "msmd_window_begin: at most 2 guidance conditions (3 entries)");
  const int d = c.d_model, Lp = c.n_prev_motions, dm = c.motion_dim;
  // at n_prev_motions = 0 the context tensors are empty (an empty torch tensor has no storage: a null pointer)
  MSMD_REQUIRE(audio && person && style && (Lp == 0 || (prev_motion && prev_audio)),
               "msmd_window_begin: null conditioning tensor");
  MSMD_REQUIRE(!c.use_indicator || indicator, "Missing indicator: the model was built with use_indicator");
  int rc;
  if ((rc = poll_overflow(m, "msmd_window_begin"))) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  m->S = S; m->NX = NX; m->E = E;
  // the conditioning the later (lazy) cache passes and every step read is copied into the handle: the caller's tensors
  // may be released as soon as this call returns, and the step graph only ever sees engine-owned addresses
  MSMD_CHECK_CUDA(cudaMemcpyAsync(m->w_audio, audio, (size_t)S * c.n_motions * d * 4, cudaMemcpyDeviceToDevice, st));
  if (Lp > 0)
    MSMD_CHECK_CUDA(cudaMemcpyAsync(m->w_prev_audio, prev_audio, (size_t)S * Lp * d * 4, cudaMemcpyDeviceToDevice, st));
  if (c.use_indicator)
    MSMD_CHECK_CUDA(cudaMemcpyAsync(m->w_ind, indicator, (size_t)S * c.n_motions * 4, cudaMemcpyDeviceToDevice, st));
  m->indicator = c.use_indicator ? m->w_ind : nullptr;
  m->window16[0] = m->window16[1] = m->window32 = false;
  if ((rc = linear_simt(person, m->dp, m->Wp, m->dp, m->bp, m->pp, d, S, d, m->dp, 0, st))) return rc;
  const int fin = dm + (c.use_indicator ? 1 : 0);
  if ((rc = linear_simt(prev_motion, dm, m->Wf, fin, m->bf_, m->pmproj, d, S * Lp, d, dm, 0, st))) return rc;
  for (int b = 0; b < c.n_basis; ++b) {
    if ((rc = linear_simt(style, c.d_style, m->Ws0[b], c.d_style, m->bs0[b], m->hid, d, S, d, c.d_style, 1, st))) return rc;
    if ((rc = linear_simt(m->hid, d, m->Ws2[b], d, m->bs2[b], m->stat + b * dm, (int64_t)c.n_basis * dm, S, dm, d, 0, st)))
      return rc;
  }
  // the cross-attention caches of the model's main arithmetic now; the other formats of a hybrid model on first use
  if (c.precision == 1) { if ((rc = window_begin_f32(m, st))) return rc; }
  else if ((rc = window_begin_16(m, c.precision == 3 ? 1 : 0, st))) return rc;
  m->window = true;
  return MSMD_OK;
}

// int64 step indices of the module-level forward -> int32, clamped to the timestep-embedding table [0, n_diff_steps]
__global__ void steps_from_i64_kernel(const int64_t* in, int* out, int S, int t_max) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < S) out[i] = (int)min((int64_t)t_max, max((int64_t)0, in[i]));
}

namespace {
// path: 0 bf16, 1 fp32-grade, 2 one-pass fp16
int check_path(const msmd_model* m, int path, const char* who) {
  const bool ok = path == 0 ? has_bf16(m->c) : (path == 1 ? has_f32(m->c) : (path == 2 ? has_fp16(m->c) : false));
  if (!ok) {
    set_error("%s: arithmetic %d (0 bf16, 1 fp32-grade, 2 fp16) is not resident in a model created with precision %d", who,
              path, m->c.precision);
    return MSMD_ERR_STATE;
  }
  return MSMD_OK;
}
int forward_path(msmd_model* m, const float* xrows, int path, cudaStream_t st) {
  int rc;
  if (path == 1) return run_forward_f32(m, xrows, st);
  const int fmt = path == 2 ? 1 : 0;
  if (!m->window16[fmt] && (rc = window_begin_16(m, fmt, st))) return rc;
  return run_forward(m, xrows, st, fmt);
}
}  // namespace

extern "C" int msmd_denoise(msmd_model* m, const float* motion, const int64_t* steps, float* out, void* stream) {
  MSMD_REQUIRE(m, "msmd_denoise: null argument");
  return msmd_denoise_ex(m, motion, steps, out, m->c.precision == 1 ? 1 : (m->c.precision == 3 ? 2 : 0), stream);
}

extern "C" int msmd_denoise_ex(msmd_model* m, const float* motion, const int64_t* steps, float* out, int precise,
                               void* stream) {
  MSMD_REQUIRE(m && motion && steps && out, "msmd_denoise: null argument");
  if (!m->window) { set_error("msmd_denoise: call msmd_window_begin first"); return MSMD_ERR_STATE; }
  MSMD_REQUIRE(m->E == 1 && m->NX == m->S, "msmd_denoise: window must be opened with NX == S, E == 1");
  int rc = check_path(m, precise, "msmd_denoise");
  if (rc) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  steps_from_i64_kernel<<<cdiv(m->S, 256), 256, 0, st>>>(steps, m->steps, m->S, m->c.n_diff_steps);
  MSMD_CHECK_LAUNCH();
  if ((rc = forward_path(m, motion, precise, st))) return rc;
  if ((rc = mix_static_launch(m->dec2, m->stat, out, m->S, m->T, m->c.motion_dim, m->c.n_basis, m->ldd, st))) return rc;
  if (precise == 1) {   // module-level parity entry: report an operand-split overflow right away (this one synchronises)
    int flag = 0;
    MSMD_CHECK_CUDA(cudaMemcpyAsync(&flag, m->overflow, sizeof(int), cudaMemcpyDeviceToHost, st));
    MSMD_CHECK_CUDA(cudaStreamSynchronize(st));
    if (flag) {
      cudaMemsetAsync(m->overflow, 0, sizeof(int), st);
      set_error("msmd_denoise: an activation left the fp16 range of the fp32-grade GEMM operand split (|x| > 65504 or NaN)");
      return MSMD_ERR_INVALID;
    }
  }
  return MSMD_OK;
}

extern "C" int msmd_denoise_parts(msmd_model* m, const float* motion, const int64_t* steps, float* dyn, float* stat,
                                  float* alphas, int precise, void* stream) {
  MSMD_REQUIRE(m && motion && steps && dyn && stat && alphas, "msmd_denoise_parts: null argument");
  if (!m->window) { set_error("msmd_denoise_parts: call msmd_window_begin first"); return MSMD_ERR_STATE; }
  MSMD_REQUIRE(m->E == 1 && m->NX == m->S, "msmd_denoise_parts: window must be opened with NX == S, E == 1");
  int rc = check_path(m, precise, "msmd_denoise_parts");
  if (rc) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  steps_from_i64_kernel<<<cdiv(m->S, 256), 256, 0, st>>>(steps, m->steps, m->S, m->c.n_diff_steps);
  MSMD_CHECK_LAUNCH();
  if ((rc = forward_path(m, motion, precise, st))) return rc;
  return split_parts_launch(m->dec2, m->stat, dyn, stat, alphas, m->S, m->T, m->c.motion_dim, m->c.n_basis, m->ldd, st);
}

extern "C" int msmd_sample_window(msmd_model* m, const float* x_T, const float* z, uint64_t seed, int cfg_independent,
                                  float scale0, float scale1, float flexibility, int t_start, int n_steps,
                                  float* x_out, float* traj, void* stream) {
  return msmd_sample_window_ex(m, x_T, z, seed, cfg_independent, scale0, scale1, flexibility, t_start, n_steps, x_out,
                               traj, nullptr, stream);
}

extern "C" int msmd_sample_window_ex(msmd_model* m, const float* x_T, const float* z, uint64_t seed, int cfg_independent,
                                     float scale0, float scale1, float flexibility, int t_start, int n_steps,
                                     float* x_out, float* traj, const msmd_sample_extras* ex, void* stream) {
  return msmd_sample_window_sched(m, x_T, z, seed, cfg_independent, scale0, scale1, flexibility, t_start, n_steps, x_out,
                                  traj, ex, nullptr, stream);
}

namespace {
// The visited steps of a respaced call (t_start and the n_steps list entries from it) and their update coefficients,
// planned in double from the loaded alpha_bars (include/msmd_b200.h, msmd_sample_schedule)
int plan_respaced(const msmd_model* m, const msmd_sample_schedule& sc, float flexibility, int t_start, int n_steps,
                  std::vector<SchedStep>& out) {
  const msmd_config& c = m->c;
  MSMD_REQUIRE(sc.timesteps && sc.n_timesteps >= 1, "msmd_sample_window: empty timestep list");
  MSMD_REQUIRE(sc.eta >= 0.f && sc.eta <= 1.f, "msmd_sample_window: eta %g outside [0, 1]", (double)sc.eta);
  MSMD_REQUIRE(sc.solver == 0 || sc.solver == 1, "msmd_sample_window: solver %d (0 DDIM, 1 DPM-Solver++(2M))", sc.solver);
  MSMD_REQUIRE(!sc.x0_prev || sc.solver == 1, "msmd_sample_window: x0_prev needs solver 1 (DPM-Solver++(2M))");
  MSMD_REQUIRE(flexibility == 0.f, "msmd_sample_window: flexibility %g has no meaning on a respaced schedule (must be 0)",
               (double)flexibility);
  const int K = sc.n_timesteps;
  const int32_t* ts = sc.timesteps;
  int pos = -1;
  for (int i = 0; i < K; ++i) {
    MSMD_REQUIRE(ts[i] >= 1 && ts[i] <= c.n_diff_steps, "msmd_sample_window: timesteps[%d] = %d outside [1, %d]", i, ts[i],
                 c.n_diff_steps);
    MSMD_REQUIRE(i == 0 || ts[i] < ts[i - 1], "msmd_sample_window: timesteps not strictly decreasing at index %d (%d after %d)",
                 i, ts[i], i ? ts[i - 1] : 0);
    if (ts[i] == t_start) pos = i;
  }
  MSMD_REQUIRE(pos >= 0, "msmd_sample_window: t_start %d is not an entry of the timestep list", t_start);
  MSMD_REQUIRE(n_steps >= 1 && pos + n_steps <= K, "msmd_sample_window: n_steps %d outside [1, %d] list entries from t_start %d",
               n_steps, K - pos, t_start);
  MSMD_REQUIRE(!sc.x0_prev || pos > 0, "msmd_sample_window: x0_prev given but t_start %d is the list's first entry", t_start);
  const std::vector<double>& ab = m->h_alpha_bars;
  const double eta = sc.eta;
  out.resize(n_steps);
  for (int i = 0; i < n_steps; ++i) {
    const int t = ts[pos + i], s = pos + i + 1 < K ? ts[pos + i + 1] : 0;
    const double A = ab[t], B = s > 0 ? ab[s] : 1.0;
    MSMD_REQUIRE(A < 1.0 && A > 0.0, "msmd_sample_window: alpha_bars[%d] = %g outside (0, 1)", t, A);
    if (sc.solver == 1) {
      // DPM-Solver++(2M) in the lambda form (include/msmd_b200.h); second order when the call has a predecessor p
      // (an earlier step of this call, or x0_prev) and s > 0
      const double al_t = std::sqrt(A), sg_t = std::sqrt(1.0 - A), lam_t = std::log(al_t / sg_t);
      double k = 0.0, M = 1.0, sigma = 0.0;   // s = 0: x_0 = D
      if (s > 0) {
        MSMD_REQUIRE(B < 1.0 && B > A, "msmd_sample_window: alpha_bars[%d] = %g outside (alpha_bars[%d], 1)", s, B, t);
        const double al_s = std::sqrt(B), sg_s = std::sqrt(1.0 - B), h = std::log(al_s / sg_s) - lam_t;
        k = sg_s / sg_t * std::exp(-eta * h);
        M = al_s * -std::expm1(-(1.0 + eta) * h);
        sigma = sg_s * std::sqrt(-std::expm1(-2.0 * eta * h));
      }
      double w1 = 1.0, w2 = 0.0;   // D = w1 x0_t + w2 x0_p
      if (s > 0 && (i > 0 || sc.x0_prev)) {
        const double Ap = ab[ts[pos + i - 1]];
        const double lam_p = std::log(std::sqrt(Ap) / std::sqrt(1.0 - Ap));
        const double h = std::log(std::sqrt(B) / std::sqrt(1.0 - B)) - lam_t, r = (lam_t - lam_p) / h;
        w1 = 1.0 + 0.5 / r;
        w2 = -0.5 / r;
      }
      // x0_t = a x_t + b out: out itself for target 'sample', (x_t - sigma_t eps_hat) / alpha_t for 'noise'
      const double a = c.target_noise ? 1.0 / al_t : 0.0, b = c.target_noise ? -sg_t / al_t : 1.0;
      // the history is written only where the next step of this call reads it
      const bool keep = i + 1 < n_steps && pos + i + 2 < K;
      out[i] = SchedStep{(float)(k + M * w1 * a), (float)(M * w1 * b), (float)sigma, (float)(M * w2),
                         keep ? (float)a : 0.f, keep ? (float)b : 0.f, t, s, i};
      continue;
    }
    const double sigma = eta * std::sqrt((1.0 - B) / (1.0 - A)) * std::sqrt(std::max(0.0, 1.0 - A / B));
    const double r = std::sqrt(std::max(0.0, 1.0 - B - sigma * sigma));
    double c0, c1;
    if (c.target_noise) {
      c0 = std::sqrt(B / A);
      c1 = r - std::sqrt(B) * std::sqrt(1.0 - A) / std::sqrt(A);
    } else {
      c0 = r / std::sqrt(1.0 - A);
      c1 = std::sqrt(B) - std::sqrt(A) * c0;
    }
    out[i] = SchedStep{(float)c0, (float)c1, (float)sigma, 0.f, 0.f, 0.f, t, s, i};
  }
  return MSMD_OK;
}
}  // namespace

extern "C" int msmd_sample_window_sched(msmd_model* m, const float* x_T, const float* z, uint64_t seed, int cfg_independent,
                                        float scale0, float scale1, float flexibility, int t_start, int n_steps,
                                        float* x_out, float* traj, const msmd_sample_extras* ex,
                                        const msmd_sample_schedule* sched, void* stream) {
  MSMD_REQUIRE(m && x_T && x_out, "msmd_sample_window: null argument");
  if (!m->window) { set_error("msmd_sample_window: call msmd_window_begin first"); return MSMD_ERR_STATE; }
  const msmd_config& c = m->c;
  std::vector<SchedStep> plan;   // respaced calls: the visited steps, in order
  if (sched) {
    int r = plan_respaced(m, *sched, flexibility, t_start, n_steps, plan);
    if (r) return r;
  } else {
    MSMD_REQUIRE(t_start >= 1 && t_start <= c.n_diff_steps && n_steps >= 1 && n_steps <= t_start,
                 "msmd_sample_window: steps %d..%d outside 1..%d", t_start, t_start - n_steps + 1, c.n_diff_steps);
    MSMD_REQUIRE(flexibility >= 0.f && flexibility <= 1.f, "msmd_sample_window: flexibility outside [0,1]");
  }
  MSMD_REQUIRE(!(ex && ex->noise_keys && z),
               "msmd_sample_window: noise_keys key the in-kernel noise and cannot be combined with an external z");
  MSMD_REQUIRE(!(sched && sched->solver == 1 && ex && ex->cumulative_static),
               "msmd_sample_window: cumulative_static is not available with solver 1 (DPM-Solver++(2M))");
  int rc;
  if ((rc = poll_overflow(m, "msmd_sample_window"))) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t n_el = (size_t)m->NX * c.n_motions * c.motion_dim;
  MSMD_CHECK_CUDA(cudaMemcpyAsync(m->xbuf, x_T, n_el * 4, cudaMemcpyDeviceToDevice, st));
  if ((rc = steps_set(m->steps, m->S, t_start, st))) return rc;

  // step schedule: t <= k32 fp32-grade, k32 < t <= k16 one-pass fp16, t > k16 the model's main 16-bit arithmetic
  int k32 = c.precision == 1 ? c.n_diff_steps : 0;
  int k16 = c.precision == 3 ? c.n_diff_steps : 0;
  if (ex && c.precision != 1) {
    k32 = ex->precise_last_steps < 0 ? c.n_diff_steps : ex->precise_last_steps;
    MSMD_REQUIRE(k32 == 0 || has_f32(c), "msmd_sample_window: precise_last_steps needs a model created with precision 2");
  }
  if (ex && c.precision != 3 && c.precision != 1) {
    k16 = ex->fp16_last_steps < 0 ? c.n_diff_steps : ex->fp16_last_steps;
    MSMD_REQUIRE(k16 == 0 || has_fp16(c), "msmd_sample_window: fp16_last_steps needs a model created with precision 2");
  }
  if (k16 < k32) k16 = k32;

  UpdateParams up{};
  up.dec = m->dec2; up.stat = m->stat; up.x = m->xbuf; up.z = z; up.traj = traj; up.steps = m->steps;
  up.alphas = m->alphas; up.alpha_bars = m->alpha_bars; up.sig_flex = m->sig_flex; up.sig_inflex = m->sig_inflex;
  up.scale0 = scale0; up.scale1 = scale1; up.flexibility = flexibility; up.seed = seed;
  up.NX = m->NX; up.E = m->E; up.T = m->T; up.L = c.n_motions; up.Lp = c.n_prev_motions; up.dm = c.motion_dim;
  up.nb = c.n_basis; up.ldd = m->ldd; up.cfg_independent = cfg_independent; up.target_noise = c.target_noise;
  up.thr = nullptr; up.tgt_dyn = nullptr; up.cum_static = nullptr; up.alpha_traj = nullptr; up.t_start = t_start;
  up.overflow = k32 > 0 ? m->overflow : nullptr;
  up.done = m->d_done; up.steps_rw = m->steps; up.S = m->S;
  bool use_dt = false;
  float dt_ratio = 0.f, dt_min = 0.f, dt_max = 0.f;
  if (ex) {
    use_dt = ex->use_dynamic_threshold != 0;
    dt_ratio = ex->dt_ratio; dt_min = ex->dt_min; dt_max = ex->dt_max;
    MSMD_REQUIRE(!use_dt || (dt_ratio >= 0.f && dt_ratio <= 1.f), "quantile() q values must be in the range [0, 1]");
    if (use_dt) up.thr = m->thr;
    up.tgt_dyn = ex->target_dynamic; up.cum_static = ex->cumulative_static; up.alpha_traj = ex->alpha_traj;
    up.noise_offset = (long long)ex->noise_clip_offset * c.n_motions * c.motion_dim;
    if (ex->noise_keys) {
      // copied into the handle: the step graph reads only engine-owned memory, and the caller may free its keys on return
      MSMD_CHECK_CUDA(cudaMemcpyAsync(m->d_keys, ex->noise_keys, (size_t)m->NX * 2 * sizeof(int64_t),
                                      cudaMemcpyDeviceToDevice, st));
      up.noise_keys = m->d_keys;
    }
    if (up.cum_static) MSMD_CHECK_CUDA(cudaMemsetAsync(up.cum_static, 0, n_el * 4, st));
  }
  if (sched) {
    // the visited steps' entries go into the engine-owned table (stream order, by value): the step graphs keep reading only
    // engine memory, so respaced and default calls of one shape share them
    if ((rc = sched_table_set(m->d_sched, plan.data(), (int)plan.size(), st))) return rc;
    up.sched = m->d_sched;
    up.hist = m->d_hist;
    // copied into the handle like noise_keys: the step graph reads only engine-owned memory
    if (sched->x0_prev) MSMD_CHECK_CUDA(cudaMemcpyAsync(m->d_hist, sched->x0_prev, n_el * 4, cudaMemcpyDeviceToDevice, st));
  }
  if ((rc = update_params_set(m->d_up, up, st))) return rc;

  // path: 0 bf16, 1 fp32-grade, 2 fp16
  auto one_step = [&](cudaStream_t s, int path) -> int {
    int r;
    if ((r = forward_path(m, m->xbuf, path, s))) return r;
    if (use_dt && (r = threshold_launch(m->dec2, m->stat, m->thr, m->S, m->T, c.n_motions, c.n_prev_motions, c.motion_dim,
                                        c.n_basis, m->ldd, dt_ratio, dt_min, dt_max, s)))
      return r;
    return update_launch(m->d_up, m->NX, c.n_motions, c.motion_dim, s);     // also advances the step index
  };

  // n consecutive steps of one 16-bit path: replays of ONE captured step (the step index lives in device memory, the
  // update parameters in m->d_up).  The instantiated graph is kept in the handle: only the first call of a given
  // (format, S, NX, E, thresholding) captures and instantiates; later calls just enqueue launches - no stream
  // creation, instantiation or synchronisation (include/msmd_b200.h: "no hidden synchronisation after *_create").
  auto run_16 = [&](int path, int n) -> int {
    if (n <= 0) return MSMD_OK;
    int r;
    const int fmt = path == 2 ? 1 : 0;
    if ((r = check_path(m, path, "msmd_sample_window"))) return r;
    if (!m->window16[fmt] && (r = window_begin_16(m, fmt, st))) return r;
    if (profiling_on() || n < 3) {  // event timing cannot live inside a graph: plain launches
      for (int i = 0; i < n; ++i)
        if ((r = one_step(st, path))) return r;
      return MSMD_OK;
    }
    const msmd_model::GraphKey key(fmt, m->S, m->NX, m->E, use_dt ? 1 : 0, dt_ratio, dt_min, dt_max);
    auto it = m->graphs.find(key);
    if (it == m->graphs.end()) {
      // first step eagerly (one-time function attributes, launch validation), then capture one step
      if ((r = one_step(st, path))) return r;
      n -= 1;
      cudaGraph_t graph = nullptr;
      cudaGraphExec_t exec = nullptr;
      MSMD_CHECK_CUDA(cudaStreamBeginCapture(m->cap_stream, cudaStreamCaptureModeThreadLocal));
      r = one_step(m->cap_stream, path);
      cudaError_t ce = cudaStreamEndCapture(m->cap_stream, &graph);
      if (r || ce != cudaSuccess) {
        if (graph) cudaGraphDestroy(graph);
        if (!r) { set_error("msmd_sample_window: graph capture failed: %s", cudaGetErrorString(ce)); r = MSMD_ERR_CUDA; }
        return r;
      }
      ce = cudaGraphInstantiate(&exec, graph, 0);
      cudaGraphDestroy(graph);
      if (ce != cudaSuccess) {
        set_error("msmd_sample_window: cudaGraphInstantiate failed: %s", cudaGetErrorString(ce));
        return MSMD_ERR_CUDA;
      }
      it = m->graphs.emplace(key, exec).first;
    }
    for (int i = 0; i < n; ++i) MSMD_CHECK_CUDA(cudaGraphLaunch(it->second, st));
    return MSMD_OK;
  };

  // executed steps are t = t_start .. t_end, or the visited entries of a respaced call; the segments are counted in t
  const int t_end = t_start - n_steps + 1;
  auto count = [&](int hi, int lo) {
    if (sched) {
      int n = 0;
      for (const SchedStep& e : plan) n += e.t <= hi && e.t >= lo;
      return n;
    }
    hi = std::min(hi, t_start); lo = std::max(lo, t_end); return hi >= lo ? hi - lo + 1 : 0;
  };
  const int n_main = count(c.n_diff_steps, k16 + 1), n_f16 = count(k16, k32 + 1), n_hi = count(k32, 1);
  if ((rc = run_16(has_bf16(c) ? 0 : 2, n_main))) return rc;
  if ((rc = run_16(2, n_f16))) return rc;
  // the last n_hi steps (t <= k32) run the fp32-grade path eagerly: each is several bf16 steps long, so launch latency
  // is hidden and a graph buys nothing
  if (n_hi > 0 && (rc = check_path(m, 1, "msmd_sample_window"))) return rc;
  for (int i = 0; i < n_hi; ++i)
    if ((rc = one_step(st, 1))) return rc;
  if (n_hi > 0 && (rc = post_overflow(m, st))) return rc;
  MSMD_CHECK_CUDA(cudaMemcpyAsync(x_out, m->xbuf, n_el * 4, cudaMemcpyDeviceToDevice, st));
  return MSMD_OK;
}

// Synchronise the stream and report a pending fp32-grade overflow (tests / callers that want the error at the call site).
extern "C" int msmd_check(msmd_model* m, void* stream) {
  MSMD_REQUIRE(m, "msmd_check: null model");
  MSMD_CHECK_CUDA(cudaStreamSynchronize(static_cast<cudaStream_t>(stream)));
  return poll_overflow(m, "msmd_check");
}
