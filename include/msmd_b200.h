/*
 * msmd_b200 — C ABI of the B200-native MSMD speech-to-face hot path.
 *
 * The reference (ubisoft/ubisoft-laforge-msmd) is pure Python/PyTorch and has no
 * FFI of its own; the drop-in boundary is its Python call surface (SURVEY.md 8(b)).
 * Each entry point below names the reference interface it replaces (file:line in
 * /root/reference).  The Python host modules in ubisoft-laforge-msmd_b200/ keep the
 * reference signatures and bind these symbols with ctypes (INTEGRATION.md).
 *
 * Conventions
 *   - every function returns 0 on success, a negative msmd_status otherwise;
 *     msmd_last_error() gives a thread-local message.  Nothing throws.
 *   - tensor arguments are contiguous row-major DEVICE pointers owned by the
 *     caller (PyTorch), fp32 unless stated.  Handles own only their packed
 *     weights and workspaces.  `stream` is a cudaStream_t passed as void*.
 *   - calls are stream-ordered; no hidden synchronisation after *_create.
 *   - a handle is bound to one device and is not thread-safe.
 */
#ifndef MSMD_B200_H
#define MSMD_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
  MSMD_OK = 0,
  MSMD_ERR_INVALID = -1,   /* bad argument (mirrors the reference's assert / ValueError) */
  MSMD_ERR_CUDA = -2,      /* CUDA runtime / driver failure */
  MSMD_ERR_STATE = -3,     /* call order (weights not loaded, window not prepared, ...) */
  MSMD_ERR_UNSUPPORTED = -4
} msmd_status;

const char* msmd_last_error(void);
/* Library/build identification: "msmd_b200 <ver> sm_100a". */
const char* msmd_version(void);

/* Optional per-kernel-class CUDA-event timing (off by default).  When enabled, instrumented
 * launches record an event pair on their own stream; msmd_profile_query synchronises those
 * events and returns the accumulated milliseconds and launch count of one kernel class
 * ("flame_fused", "gemm_bf16", ...).  Launches inside a CUDA-graph capture are not timed. */
int msmd_profile_enable(int on);
int msmd_profile_reset(void);
int msmd_profile_query(const char* name, double* total_ms, int64_t* launches);
/* All classes as text lines "name total_ms launches" (NUL-terminated, truncated to cap). */
int msmd_profile_dump(char* buf, int64_t cap);

/* ------------------------------------------------------------------------- *
 * Rotation conversions — utils/rotation_conversions.py:38-569
 * One fused elementwise kernel per conversion; `n` rotations; in/out packed
 * [n, k] fp32 with k = 3 (axis-angle, euler), 4 (quaternion wxyz), 6, or 9
 * (row-major 3x3).  `convention` encodes an Euler convention "ABC" as
 * a*9 + b*3 + c with X=0,Y=1,Z=2 (ignored by non-Euler kinds).
 * ------------------------------------------------------------------------- */
typedef enum {
  MSMD_ROT_QUAT_TO_MATRIX = 0,        /* quaternion_to_matrix        :38  */
  MSMD_ROT_MATRIX_TO_QUAT = 1,        /* matrix_to_quaternion        :100 */
  MSMD_ROT_EULER_TO_MATRIX = 2,       /* euler_angles_to_matrix      :151 */
  MSMD_ROT_MATRIX_TO_EULER = 3,       /* matrix_to_euler_angles      :219 */
  MSMD_ROT_AA_TO_QUAT = 4,            /* axis_angle_to_quaternion    :450 */
  MSMD_ROT_QUAT_TO_AA = 5,            /* quaternion_to_axis_angle    :481 */
  MSMD_ROT_AA_TO_MATRIX = 6,          /* axis_angle_to_matrix        :418 */
  MSMD_ROT_MATRIX_TO_AA = 7,          /* matrix_to_axis_angle        :434 */
  MSMD_ROT_6D_TO_MATRIX = 8,          /* rotation_6d_to_matrix       :513 */
  MSMD_ROT_MATRIX_TO_6D = 9,          /* matrix_to_rotation_6d       :538 */
  MSMD_ROT_AA_TO_6D = 10,             /* axis_angle_to_rotation_6d   :555 */
  MSMD_ROT_STANDARDIZE_QUAT = 11,     /* standardize_quaternion      :326 */
  MSMD_ROT_QUAT_INVERT = 12,          /* quaternion_invert           :380 */
  MSMD_ROT_EULER_TO_AA = 13,          /* fused euler->matrix->axis-angle (decode adapter, SURVEY 8(f)-1) */
  MSMD_ROT_RODRIGUES = 14             /* utils/lbs.py:270 batch_rodrigues (||r+1e-8|| quirk) */
} msmd_rot_kind;

int msmd_rot_convert(int kind, const float* in, float* out, int64_t n, int convention, void* stream);

/* Binary quaternion ops — quaternion_raw_multiply :341, quaternion_multiply :362,
 * quaternion_apply :396.  a,b already broadcast to [n,4] / [n,3] by the host. */
typedef enum {
  MSMD_QUAT_RAW_MULTIPLY = 0,
  MSMD_QUAT_MULTIPLY = 1,
  MSMD_QUAT_APPLY = 2
} msmd_quat_binop;

int msmd_quat_binary(int op, const float* a, const float* b, float* out, int64_t n, void* stream);

/* ------------------------------------------------------------------------- *
 * Linear layer on the tensor cores — every nn.Linear on the path (model.py:931-961,
 * nn.TransformerDecoderLayer / nn.MultiheadAttention projections, style_encoder.py:137-175,
 * HF encoder projections):   out[M,N] = act(x[M,K] . w[N,K]^T + bias[N]) (+ aux[M,N])
 *   mode 0: x, w bf16; one tcgen05 kind::f16 pass, fp32 accumulation in TMEM.
 *   mode 1: fp32-grade: x/x_lo and w/w_lo are tf32 hi/lo splits (msmd_split_tf32); three
 *           kind::tf32 passes (hi*hi + hi*lo + lo*hi).  out/aux fp32.
 *   mode 2: fp32-grade, faster: x/x_lo and w/w_lo are fp16 two-term splits (msmd_split_f16: x = hi + 2^-11 lo,
 *           22 mantissa bits; |x| < 65504); three kind::f16 passes, cross terms rescaled in the epilogue.
 *   mode 3: x, w and (16-bit) out IEEE fp16; one kind::f16 pass - the cost of mode 0 with 11 mantissa bits.
 *   ld* are row strides in elements (rows must be 16-byte multiples apart); act 0 none, 1 GELU(erf);
 *   out_f32 / aux_f32 select fp32 (1) or bf16 (0) for out / aux.
 * ------------------------------------------------------------------------- */
int msmd_linear(int mode, const void* x, const void* x_lo, const void* w, const void* w_lo,
                const float* bias, const void* aux, void* out, int M, int N, int K, int64_t ldx,
                int64_t ldw, int64_t ldo, int64_t ld_aux, int out_f32, int aux_f32, int act, void* stream);
int msmd_split_tf32(const float* x, float* hi, float* lo, int64_t n, void* stream);
int msmd_split_f16(const float* x, void* hi, void* lo, int64_t n, void* stream);   /* hi, lo: __half[n] */

/* ------------------------------------------------------------------------- *
 * Denoiser + sampler — model.py:820-996 (DenoisingNetwork_MSMD), :282-440 (MSMD.sample),
 * :20-71 (DiffusionSchedule).
 *
 * A "sequence" is one row of the reference's concatenated CFG batch (model.py:368-374):
 * S = E * NX sequences for NX clips and E classifier-free-guidance entries, sequence
 * s = e * NX + n.  All sequences of a window share the step index.
 * ------------------------------------------------------------------------- */
typedef struct {
  int n_motions;        /* L   = 100 */
  int n_prev_motions;   /* Lp  = 10  */
  int d_model;          /* 512 */
  int n_heads;          /* 8   */
  int n_layers;         /* 8   */
  int d_ff;             /* mlp_ratio * d_model = 2048 */
  int d_style;          /* 256 */
  int d_shape;          /* 100 */
  int motion_dim;       /* 67  */
  int n_basis;          /* 4;  >= 1 (the reference has no result for num_of_basis = 0), motion_dim + n_basis <= 80 */
  int n_diff_steps;     /* 500 */
  int use_indicator;    /* 1   */
  int align_mask_width; /* 1; >= 0.  Band of the cross-attention mask: motion token i sees memory tokens
                         * [i-1-(w-1), i-1+(w-1)], the person token all of them; 0 = no mask.  Width 1 caches the motion
                         * rows' cross attention per window; any other width runs the banded attention on every step */
  int target_noise;     /* 0: network predicts the sample (args.target == 'sample'), 1: the noise */
  int max_seqs;         /* capacity in sequences (E * clips); workspaces are sized for it at create */
  int precision;        /* 0: bf16 tensor-core GEMMs (fp32 accumulate, fp32 LayerNorm/softmax statistics);
                         * 1: fp32-grade only — fp32 activations, 3-pass fp16-split tcgen05 GEMMs (error ~1e-6), exact erf GELU;
                         * 2: hybrid — bf16, one-pass fp16 and fp32-grade weights/workspaces all resident, selectable per
                         *    call (msmd_denoise_ex) or per step (msmd_sample_extras.fp16_last_steps / precise_last_steps);
                         * 3: one-pass fp16 only (bf16's cost, x0_hat error 8e-4 instead of 6.5e-3; |activation| < 65504) */
} msmd_config;

typedef struct msmd_model msmd_model;

int msmd_create(const msmd_config* cfg, int device, msmd_model** out);
void msmd_destroy(msmd_model* m);

/* Weights by state_dict key (SURVEY App. E): "denoising_net.*" and "diffusion_sched.*" entries of
 * MSMD.state_dict() (model.py:115-137, :855-906).  fp32 data, host or device pointers; copied and
 * re-packed (bf16 casts, transposes, the 501-row timestep-embedding table) — the caller keeps its tensors. */
int msmd_load_weights(msmd_model* m, const char* const* names, const void* const* data,
                      const int64_t* numel, int n);

/* Per-window, step-invariant work (SURVEY section 0): memory K/V projections of every layer, the
 * cross-attention output of motion rows (== out_proj(v_proj(audio[i-1])) under the width-1 alignment
 * mask; other widths attend on every step), person_proj, previous-motion projection, static-basis MLPs.
 * Arguments are exactly the conditioning tensors of DenoisingNetwork_MSMD.forward (model.py:914):
 *   audio [S,L,d], person [S,d_shape+d_style], style [S,d_style], prev_motion [S,Lp,dm],
 *   prev_audio [S,Lp,d], indicator [S,L] or NULL.  S = E*NX.  Everything later calls need is copied or projected
 * into the handle in stream order: the caller may release its tensors when the call returns. */
int msmd_window_begin(msmd_model* m, const float* audio, const float* person, const float* style,
                      const float* prev_motion, const float* prev_audio, const float* indicator,
                      int S, int NX, int E, void* stream);

/* One forward of the denoising network (model.py:914-996) for module-level parity.
 * Needs msmd_window_begin(..., S, NX=S, E=1).  motion [S,L,dm]; steps [S] int64; out [S,Lp+L,dm]. */
int msmd_denoise(msmd_model* m, const float* motion, const int64_t* steps, float* out, void* stream);
/* Same, choosing the arithmetic: precise = 0 bf16 (precision 0/2), 1 fp32-grade (precision 1/2), 2 one-pass fp16
 * (precision 2/3).  msmd_denoise picks the model's main arithmetic.  Step indices are clamped to [0, n_diff_steps].
 * precise = 1 synchronises `stream` to report an fp16-range overflow of the operand split at the call site. */
int msmd_denoise_ex(msmd_model* m, const float* motion, const int64_t* steps, float* out, int precise, void* stream);
/* keep_separate=True of DenoisingNetwork_MSMD.forward (model.py:914,972-973): the un-mixed parts
 *   dyn [S,Lp+L,dm], stat [S,Lp+L,n_basis,dm] (static-basis MLP outputs tiled over the rows), alphas [S,Lp+L,n_basis]. */
int msmd_denoise_parts(msmd_model* m, const float* motion, const int64_t* steps, float* dyn, float* stat, float* alphas,
                       int precise, void* stream);

/* Ancestral sampling loop of MSMD.sample (model.py:377-435) for the current window, steps
 * t = t_start .. t_start-n_steps+1.  One step is captured as a CUDA graph the first time a (format, S, NX, E) shape
 * is seen and the instantiated graph is kept in the handle: later calls only enqueue launches (no capture, no
 * instantiation, no stream creation, no synchronisation) and return before the stream has drained.
 *   x_T [NX,L,dm] start state (state at t_start);  z [T+1,NX,L,dm] noise indexed by t or NULL
 *   (-> in-kernel Philox keyed by `seed`); cfg_independent selects 'independent' vs 'incremental';
 *   scale0/scale1 = guidance scales of entries 1 and 2; x_out [NX,L,dm];
 *   traj [T+1,NX,L,dm] or NULL receives x_{t-1} at index t-1 for every executed step. */
int msmd_sample_window(msmd_model* m, const float* x_T, const float* z, uint64_t seed, int cfg_independent,
                       float scale0, float scale1, float flexibility, int t_start, int n_steps,
                       float* x_out, float* traj, void* stream);

/* Optional extras of the sampling loop.
 *   dynamic thresholding (model.py:396-402): per sequence, clamp the network output to +-s with
 *     s = clamp(quantile(|x0_hat[:, -L:]|, dt_ratio), dt_min, dt_max)   (torch.quantile, 'linear');
 *   separate outputs of MSMD.sample_separate (model.py:442-651, alpah_t_modification = None):
 *     target_dynamic [NX,L,dm] (CFG-combined dynamic part of the last executed step),
 *     cumulative_static [NX,L,dm] (sum over steps of c1(t) * CFG-combined static part; zeroed by the call),
 *     alpha_traj [n_steps,NX,L,n_basis] (CFG-combined alphas, first executed step first).
 * Any output pointer may be NULL. */
typedef struct {
  int use_dynamic_threshold;
  float dt_ratio, dt_min, dt_max;
  float* target_dynamic;
  float* cumulative_static;
  float* alpha_traj;
  int precise_last_steps; /* hybrid schedule (precision 2): steps with t <= precise_last_steps run the fp32-grade
                           * path, earlier (noisier) steps a 16-bit path; < 0 = every step.  Ignored (all steps
                           * precise) when precision == 1; must be 0 when precision == 0 or 3.  An fp16-range overflow
                           * of the operand split poisons x_out with NaN and is reported by the NEXT call on the
                           * handle (or msmd_check) - this call does not synchronise. */
  int fp16_last_steps;    /* hybrid schedule (precision 2): steps with precise_last_steps < t <= fp16_last_steps run the
                           * one-pass fp16 path, earlier steps bf16; < 0 = every step.  Must be 0 when precision == 0. */
  int64_t noise_clip_offset; /* in-kernel Philox noise (z == NULL) is keyed by (seed, t, GLOBAL element index): clip n of
                           * this call draws the noise of global clip noise_clip_offset + n, so a clip's codes do not
                           * depend on how the clips are partitioned over calls / GPUs (SURVEY 8(e)). */
  const int64_t* noise_keys;  /* device [NX][2] or NULL: clip n of this call draws the in-kernel Philox noise of
                               * (seed = noise_keys[n][0], global clip id = noise_keys[n][1]) instead of
                               * (seed, noise_clip_offset + n), so one call can mix clips of different windows / seeds.
                               * Copied into the handle in stream order (the caller may free it when the call returns);
                               * not allowed together with z. */
} msmd_sample_extras;

int msmd_sample_window_ex(msmd_model* m, const float* x_T, const float* z, uint64_t seed, int cfg_independent,
                          float scale0, float scale1, float flexibility, int t_start, int n_steps,
                          float* x_out, float* traj, const msmd_sample_extras* extras, void* stream);

/* Respaced (DDIM) schedule of the sampling loop: the strictly decreasing HOST list of visited timesteps
 * t_1 > ... > t_K in [1, n_diff_steps], and eta in [0, 1].  With s the successor of t in the list (0 after the last
 * entry), A = alpha_bars[t], B = alpha_bars[s] (alpha_bars[0] = 1) and
 *   sigma = eta sqrt((1 - B) / (1 - A)) sqrt(1 - A / B),  r = sqrt(max(0, 1 - B - sigma^2)),
 * a step is x_s = k x_t + (sqrt(B) - sqrt(A) k) x0_hat + sigma z_t with k = r / sqrt(1 - A)       (target 'sample')
 *        or x_s = sqrt(B / A) x_t + (r - sqrt(B) sqrt(1 - A) / sqrt(A)) eps_hat + sigma z_t           (target 'noise').
 * z_t is the noise of step t of the default loop (z[t], or the in-kernel Philox stream keyed by t) and is drawn only
 * when s > 0.  The list is read on the host during the call and may be freed on return.
 *
 * solver 1 is DPM-Solver++(2M) (its SDE variant for eta > 0; this eta is not DDIM's).  With alpha = sqrt(alpha_bar),
 * sigma = sqrt(1 - alpha_bar), lambda = log(alpha / sigma), p the entry executed before t, h = lambda_s - lambda_t and
 * r = (lambda_t - lambda_p) / h, a step is
 *   D   = x0_t + (x0_t - x0_p) / (2 r)    (D = x0_t when there is no p, and on the step to s = 0)
 *   x_s = (sigma_s / sigma_t) e^{-eta h} x_t + alpha_s (1 - e^{-(1 + eta) h}) D + sigma_s sqrt(1 - e^{-2 eta h}) z_t
 * where x0 is the CFG-combined, thresholded data prediction (x0 = (x_t - sigma_t eps_hat) / alpha_t for target
 * 'noise'); z_t is drawn as for solver 0.  A first-order step has DDIM's coefficients at eta = 0 and at eta = 1.
 * The engine keeps x0 of the last executed step per row; a call starts without one, so its first step is first
 * order unless x0_prev is given.
 *   solver:  0 = DDIM (zero-initialised callers), 1 = DPM-Solver++(2M); anything else is MSMD_ERR_INVALID.
 *   x0_prev: device [NX, L, dm] or NULL: x0 of the list entry before t_start, so a call that starts mid-list takes its
 *            first step at second order.  Copied into the handle in stream order (the caller may free it on return).
 *            MSMD_ERR_INVALID with solver 0 and when t_start is the list's first entry.
 * Solver 1 together with extras->cumulative_static is MSMD_ERR_INVALID. */
typedef struct {
  const int32_t* timesteps;
  int n_timesteps;
  float eta;
  int solver;
  const float* x0_prev;
} msmd_sample_schedule;

/* msmd_sample_window_ex on a respaced schedule (sched = NULL: the default loop t = t_start .. t_start - n_steps + 1).
 * t_start must be an entry of the list and n_steps counts list entries from there.  flexibility must be 0.  traj
 * receives x_s at index s; extras->alpha_traj row i is the i-th executed step; extras->cumulative_static sums the
 * output coefficient times the static part.  The hybrid precision schedule keeps its meaning in t: visited steps with
 * t <= precise_last_steps run fp32-grade, t <= fp16_last_steps fp16.  Step graphs are shared with the default loop. */
int msmd_sample_window_sched(msmd_model* m, const float* x_T, const float* z, uint64_t seed, int cfg_independent,
                             float scale0, float scale1, float flexibility, int t_start, int n_steps,
                             float* x_out, float* traj, const msmd_sample_extras* extras,
                             const msmd_sample_schedule* sched, void* stream);

/* Synchronise `stream` and report a pending fp32-grade operand-split overflow of an earlier call on this handle. */
int msmd_check(msmd_model* m, void* stream);

/* ------------------------------------------------------------------------- *
 * Style encoder — style_encoder.py:119-213 (StyleEncoder_VAE2.forward / .sample)
 * motion [N,L,d_in] -> mu, logvar [N,d_style]; style = mu + eps * exp(0.5 logvar) with the
 * caller's eps [N,d_style] (NULL -> style = mu).  Any of the three outputs may be NULL.
 * Weights by state_dict key (SURVEY App. E, "StyleEncoder_VAE2").  L <= 112 frames.
 * ------------------------------------------------------------------------- */
typedef struct msmd_style msmd_style;
int msmd_style_create(int d_in, int d_model, int d_style, int max_clips, int max_len, int device,
                      msmd_style** out);
void msmd_style_destroy(msmd_style* m);
int msmd_style_load_weights(msmd_style* m, const char* const* names, const void* const* data,
                            const int64_t* numel, int n);
int msmd_style_encode(msmd_style* m, const float* motion, int N, int L, const float* eps, float* style_out,
                      float* mu_out, float* logvar_out, void* stream);

/* ------------------------------------------------------------------------- *
 * Audio encoder — utils/hubert.py:13-51, utils/wav2vec2.py:71-119 (HF Hubert / Wav2Vec2 *base*
 * forward with the reference's 50 fps -> output_fps resampling) and model.py:250-264
 * (MSMD.extract_audio_feature: encode at 2L frames, 2:1 linear resample, Linear 768 -> d).
 * wav [N, n_samples] fp32 16 kHz (un-padded: pad_audio, model_common.py:110-123, is folded into the
 * first conv's loads).  hidden_out [N, frame_num, 768] (last_hidden_state) and/or
 * feat_out [N, feat_frames, d_out]; either may be NULL.
 * Weights: "audio_encoder.*" (HF key names, SURVEY App. E) and optionally "audio_feature_map.*".
 * ------------------------------------------------------------------------- */
typedef struct msmd_audio msmd_audio;
int msmd_audio_create(int max_clips, int max_samples, int d_out, int device, msmd_audio** out);
void msmd_audio_destroy(msmd_audio* m);
int msmd_audio_load_weights(msmd_audio* m, const char* const* names, const void* const* data,
                            const int64_t* numel, int n);
int msmd_audio_encode(msmd_audio* m, const float* wav, int N, int n_samples, int output_fps, int frame_num,
                      float* hidden_out, int feat_frames, float* feat_out, void* stream);

/* ------------------------------------------------------------------------- *
 * Clip front-end of the inference driver (the numpy stages between file I/O and the encoders)
 *   msmd_audio_normalize: inference.py:234   out = (x - mean(x)) / (std(x) + 1e-5) per clip (population std);
 *                         in/out [n_clips, n_samples] fp32, may alias.
 *   msmd_resample_linear: inference.py:158-171   scipy interp1d(kind='linear', axis=0) from
 *                         np.linspace(0,1,rows_in) onto np.linspace(0,1,rows_out); in [rows_in, cols], out [rows_out, cols].
 * ------------------------------------------------------------------------- */
int msmd_audio_normalize(const float* in, float* out, int n_clips, int64_t n_samples, void* stream);
int msmd_resample_linear(const float* in, float* out, int rows_in, int rows_out, int cols, void* stream);

/* ------------------------------------------------------------------------- *
 * FLAME decode — utils/flame.py:180-244 (FLAME.forward) -> utils/lbs.py:141-223 (lbs)
 *
 * msmd_flame_create packs the static bases once:
 *   v_template [V,3], shapedirs [V,3,NB], posedirs [(NJ-1)*9, V*3],
 *   J_regressor [NJ,V], parents [NJ] (int64, parents[0] = -1), lbs_weights [V,NJ].
 *   Pointers may be host or device (copied with cudaMemcpyDefault).
 * msmd_flame_decode runs F1-F6 of SURVEY 2.4 fused:
 *   betas [B,NB]; pose [B,NJ*3] axis-angle if pose2rot else [B,NJ*9] matrices;
 *   verts_out [B,V,3]; joints_out [B,NJ,3] or NULL.
 * `impl`: 0 = default (tensor-core path), 1 = CUDA-core reference path (debug).
 * ------------------------------------------------------------------------- */
typedef struct msmd_flame msmd_flame;

int msmd_flame_create(const float* v_template, const float* shapedirs, const float* posedirs,
                      const float* J_regressor, const int64_t* parents, const float* lbs_weights,
                      int V, int NB, int NJ, int device, msmd_flame** out);
int msmd_flame_decode(msmd_flame* fh, const float* betas, const float* pose, int pose2rot,
                      int64_t B, float* verts_out, float* joints_out, int impl, void* stream);
void msmd_flame_destroy(msmd_flame* fh);

/* Barycentric landmarks — utils/lbs.py:102-138 (vertices2landmarks).
 * verts [B,V,3]; faces [F,3] int64; lmk_faces_idx [B,L] int64; bary [B,L,3]; out [B,L,3]. */
int msmd_vertices2landmarks(const float* verts, const int64_t* faces, const int64_t* lmk_faces_idx,
                            const float* bary, int64_t B, int V, int L, float* out, void* stream);

/* Dynamic face-contour row per frame — utils/flame.py:126-172 (_find_dynamic_lmk_idx_and_bcoords)
 * with utils/lbs.py:26-32 (rot_mat_to_euler).  full_pose [B,NJ*3] (or [B,NJ*9] if !pose2rot);
 * neck_chain [n_chain] int64 joint ids (device); out_idx [B] int64 in [0,78]. */
int msmd_flame_contour_index(const float* full_pose, int pose2rot, int NJ, const int64_t* neck_chain,
                             int n_chain, int64_t B, int64_t* out_idx, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MSMD_B200_H */
