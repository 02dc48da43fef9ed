// Non-GEMM kernels of the denoiser / sampler (model.py:914-996, :377-435): declarations.
#pragma once
#include "common.cuh"
#include <cuda_bf16.h>

namespace msmd {

using bf16 = __nv_bfloat16;

// out[r,c] = act(b[c] + sum_k x[r,k] W[c,k])  — small fp32 linears (step-invariant precompute only)
int linear_simt(const float* x, int64_t ldx, const float* W, int64_t ldw, const float* b, float* out, int64_t ldo, int R,
                int C, int K, int act, cudaStream_t st);

// fp32 -> bf16 cast of a [rows, cols] block into a strided destination
int cast_rows_bf16(const float* src, int64_t lds, bf16* dst, int64_t ldd, int64_t rows, int cols, cudaStream_t st);

// 16-bit activation buffers are typed bf16* whatever their storage format; `fp16` != 0 selects IEEE half storage
// (the sampler's intermediate-precision steps), 0 bfloat16.
// memory = cat(prev_audio [S,Lp,d], audio [S,L,d]) -> 16-bit [S, Lp+L, d]
int build_memory_h16(const float* prev_audio, const float* audio, bf16* mem, int S, int Lp, int L, int d, int fp16,
                     cudaStream_t st);

struct EmbedParams {
  // rows 0..Lp of every sequence (step-dependent only through the timestep embedding)
  const float* pp;        // [S, d]   person_proj(person) (per window)
  const float* temb;      // [T+1, d] diff_step_map(TE.pe) table
  const float* pmproj;    // [S, Lp, d] feature_proj([prev_motion, 0]) (per window)
  const float* PE;        // [1+Lp+L, d]
  const int* steps;       // [S]
  // rows Lp+1.. : feature_proj([x_t, indicator]) + PE
  const float* x;         // [NX, L, dm]
  const float* indicator; // [S, L] or null (-> no indicator column)
  const float* WfT;       // [dm+1, d] feature_proj weight transposed (k-major), fp32
  const float* bf;        // [d]
  const void* Wf16;       // [2][d][80] fp16: hi | lo halves of feature_proj.weight[:, :dm] (K zero-padded to 80), or null
                          // (-> the CUDA-core kernel); the tensor-core embedding (embed_x_mma_kernel) needs d = 512, dm <= 80
  bf16* out;              // [S, 1+Lp+L, d]
  int S, NX, E, Lp, L, d, dm;
  int fp16;               // storage format of `out`
};
int embed_launch(const EmbedParams& p, cudaStream_t st);

// y [M,512] fp32 -> LayerNorm(g1,b1); rows with (token != 0): + add[(seq, token-1)] then LayerNorm(g2,b2) (optional)
// -> out bf16 [M,512]; token-0 rows: LN1 only, written to x0 [S,512] (and NOT to out) when x0 != null.
struct LnParams {
  const bf16* y;            // [M, d] sub-layer output (GEMM epilogue writes bf16)
  const bf16* resid;        // [M, d] residual stream added to y before the first LayerNorm (may alias out), or null
  const float* g1; const float* b1;
  const bf16* add;          // [S, T-1, d] or null
  const float* g2; const float* b2;   // used iff add != null
  bf16* out;                // [M, d]
  bf16* x0;                 // [S, d] or null
  int skip_tok0;            // do not write token-0 rows at all (they are produced by the person-token stream)
  int M, T, d;
  int fp16;                 // storage format of y / resid / add / out / x0
};
int ln_launch(const LnParams& p, cudaStream_t st);
// row-0 finish: LayerNorm(y0 [S,d]; g,b) -> out[s*T + 0]
// LayerNorm(y0 + resid0) of the S person-token rows -> out[s*T + 0] (if out) and compact out_c[s] (if out_c)
int ln_row0_launch(const bf16* y0, const bf16* resid0, const float* g, const float* b, bf16* out, bf16* out_c, int S,
                   int T, int d, int fp16, cudaStream_t st);

// row-0 cross attention: q0 [S,d]; kv [S*Tk, 2d] (k|v) -> ctx0 [S,d]
int cross_attn_row0_launch(const bf16* q0, const bf16* kv, bf16* ctx0, int S, int Tk, int H, int fp16, cudaStream_t st);


// One visited step t of a respaced schedule (msmd_sample_window_sched): x_s = c0 x_t + c1 out + c2 h_p + sigma z_t,
// where out is the network output (x0_hat or eps_hat), h_p the data prediction of the previous step (history buffer;
// c2 = 0: not read), s = next (0 after the last entry) and ord = position from the call's t_start.  b != 0: the step
// writes its own data prediction h_t = a x_t + b out to the history for the next step.  DDIM steps have c2 = a = b = 0.
struct SchedStep {
  float c0, c1, sigma, c2, a, b;
  int t, next, ord;
};

struct UpdateParams {
  const float* dec;       // [S, T, ldd] fp32: motion_dec output (dm dynamic + nb alphas)
  const float* stat;      // [S, nb, dm]
  float* x;               // [NX, L, dm]  in/out
  const float* z;         // [Tsteps+1, NX, L, dm] or null
  float* traj;            // [Tsteps+1, NX, L, dm] or null (writes index t-1)
  const int* steps;       // [S] (all equal in sampling mode)
  const float* alphas; const float* alpha_bars; const float* sig_flex; const float* sig_inflex;  // [Tsteps+1]
  float scale0, scale1, flexibility;
  unsigned long long seed;
  int NX, E, T, L, Lp, dm, nb, ldd;
  int cfg_independent, target_noise;
  // optional (msmd_sample_extras): dynamic thresholding (model.py:396-402) and the separate outputs of
  // MSMD.sample_separate (model.py:442-651)
  const float* thr;       // [S] per-sequence clamp of the network output, or null
  float* tgt_dyn;         // [NX, L, dm] CFG-combined dynamic part of the LAST executed step, or null
  float* cum_static;      // [NX, L, dm] += c1 * CFG-combined static part, or null
  float* alpha_traj;      // [n_steps, NX, L, nb] CFG-combined alphas per executed step (index t_start - t), or null
  int t_start;
  unsigned int* done;     // block-completion counter (zeroed): the last block writes steps_rw[0..S) = t - 1, or null
  int* steps_rw;          // [S] same array as `steps`
  int S;
  long long noise_offset; // added to the element index that keys the in-kernel Philox noise (= global clip id * L * dm)
  const int* overflow;    // fp32-grade steps: device flag raised by the operand split; non-zero poisons x with NaN
  const long long* noise_keys;  // [NX][2] (seed, global clip id) per clip, or null (-> seed, noise_offset); engine-owned
  // respaced schedule: [n_diff_steps + 1] indexed by t (engine-owned), or null (-> the posterior step t -> t - 1).  When
  // set, the step takes its coefficients from sched[t], draws noise iff next > 0, writes traj at next and alpha_traj at
  // ord, and advances steps_rw to next
  const SchedStep* sched;
  // [NX, L, dm] data prediction of the last executed step (engine-owned), read where sched[t].c2 != 0 and written where
  // sched[t].b != 0, element by element by the same thread
  float* hist;
};
// per-sequence threshold s = clamp(quantile(|x0_hat[:, -L:]|, ratio), lo, hi) -> thr[S] (torch.quantile 'linear')
int threshold_launch(const float* dec, const float* stat, float* thr, int S, int T, int L, int Lp, int dm, int nb, int ldd,
                     float ratio, float lo, float hi, cudaStream_t st);
// the parameter block is read from DEVICE memory (d_p), written by update_params_set in stream order
int update_params_set(UpdateParams* d_dst, const UpdateParams& p, cudaStream_t st);
int update_launch(const UpdateParams* d_p, int NX, int L, int dm, cudaStream_t st);
// scatter n host entries into table[entry.t], in stream order (by-value kernel arguments: the host array may be freed on
// return, and nothing synchronises)
int sched_table_set(SchedStep* table, const SchedStep* h, int n, cudaStream_t st);
int steps_set(int* steps, int S, int value, cudaStream_t st);

// out[S, T-1... ] : x̂0 per sequence (module-level parity): dyn + static mix for ALL Lp+L rows -> [S, T-1, dm]
int mix_static_launch(const float* dec, const float* stat, float* out, int S, int T, int dm, int nb, int ldd, cudaStream_t st);

// the whole person-token cross-attention block (q-proj, attention over the memory, out-proj, residual, norm2) as one
// cluster kernel (row0_fused.cu): x0c [S,512] -> x[s*T + 0]
int row0_fused_launch(const bf16* x0c, const bf16* Wq, const float* bq, const bf16* kv, const bf16* Wo, const float* bo,
                      const float* g, const float* be, bf16* x, int S, int T, int Tk, int H, int d, int fp16, cudaStream_t st);

// keep_separate outputs (model.py:972-973): dyn [S,T-1,dm], sta [S,T-1,nb,dm] (tiled), alphas [S,T-1,nb]
int split_parts_launch(const float* dec, const float* stat, float* dyn, float* sta, float* alphas, int S, int T, int dm,
                       int nb, int ldd, cudaStream_t st);

// tcgen05 self-attention (attn_tc.cu) over T <= 112 tokens, head dim 64: qkv [S*T, 3*d] (q|k|v) -> ctx [S*T, d], 16-bit storage
int self_attn_tc_launch(const bf16* qkv, bf16* ctx, int S, int T, int H, int fp16, cudaStream_t st);
// the same kernel in its cross-attention mode: q [S*T, d], kv [S*Tk, 2d] (k|v, the per-window cache) -> ctx [S*T, d] under
// the alignment band of `width` (token 0 sees every key; token r >= 1 the keys c with |c - (r-1)| <= width-1; 0 = no band)
int cross_attn_tc_launch(const bf16* q, const bf16* kv, bf16* ctx, int S, int T, int Tk, int H, int width, int fp16,
                         cudaStream_t st);

// ---- fp32-grade variants (denoiser_f32.cu) ----
int embed_f32_launch(const EmbedParams& p, float* out, cudaStream_t st);
int ln_f32_launch(const float* y, const float* resid, const float* g1, const float* b1, const float* add, const float* g2,
                  const float* b2, float* out, float* x0, int M, int T, cudaStream_t st);
int ln_row0_f32_launch(const float* y0, const float* r0, const float* g, const float* b, float* out, int S, int T,
                       cudaStream_t st);
int self_attn_f32_launch(const float* qkv, float* ctx, int S, int T, int H, cudaStream_t st);
int cross_attn_f32_launch(const float* q, const float* kv, float* ctx, int S, int T, int Tk, int H, int width,
                          cudaStream_t st);
int cross_attn_row0_f32_launch(const float* q0, const float* kv, float* ctx0, int S, int Tk, int H, cudaStream_t st);
int build_memory_f32(const float* prev_audio, const float* audio, float* mem, int S, int Lp, int L, int d, cudaStream_t st);
int split_tf32(const float* x, float* hi, float* lo, int64_t n, cudaStream_t st);   // gemm_tc.cu

}  // namespace msmd
