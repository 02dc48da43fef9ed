"""Drop-in for /root/reference/model.py on the inference path.

Same constructors (an ``argparse.Namespace`` of hyper-parameters), same ``state_dict`` keys and shapes
(SURVEY App. E) and same call signatures for ``get_diffusion_model``, ``DiffusionSchedule``,
``DenoisingNetwork_MSMD.forward``, ``MSMD.sample`` and ``MSMD.extract_audio_feature``; the modules
only HOLD parameters - every forward runs in the CUDA engine behind the C ABI (csrc/denoiser*.cu,
csrc/gemm_tc.cuh).  Training-only code paths of the reference (MSMD.forward's noising / CFG dropout,
model.py:146-248) are out of scope and raise.
"""
import math
from fractions import Fraction

import torch
import torch.nn as nn

from . import _lib
from ._engine import DenoiserEngine, PRECISIONS
from .utils.model_common import PositionalEncoding, enc_dec_mask


def get_diffusion_model(args, device='cuda'):
    """model.py:7-17."""
    if not hasattr(args, 'style_enc_ckpt'):
        args.style_enc_ckpt = None
    regularizer = getattr(args, 'regularize_alpha', "None")
    return MSMD(args, device, True, use_head_alpha=False, regularize_alpha=regularizer)


class DiffusionSchedule(nn.Module):
    """model.py:20-71.  Buffers are built with the same fp32 torch operations (bit-identical tables);
    a loaded checkpoint overwrites them anyway."""

    def __init__(self, num_steps, mode='linear', beta_1=1e-4, beta_T=0.02, s=0.008):
        super().__init__()
        if mode == 'linear':
            betas = torch.linspace(beta_1, beta_T, num_steps)
        elif mode == 'quadratic':
            betas = torch.linspace(beta_1 ** 0.5, beta_T ** 0.5, num_steps) ** 2
        elif mode == 'sigmoid':
            betas = torch.sigmoid(torch.linspace(-5, 5, num_steps)) * (beta_T - beta_1) + beta_1
        elif mode == 'cosine':
            x = torch.linspace(0, num_steps, num_steps + 1)
            ab = torch.cos(((x / num_steps) + s) / (1 + s) * torch.pi * 0.5) ** 2
            ab = ab / ab[0]
            betas = torch.clip(1 - (ab[1:] / ab[:-1]), 0.0001, 0.999)
        else:
            raise ValueError(f'Unknown diffusion schedule {mode}!')
        betas = torch.cat([torch.zeros(1), betas], dim=0)
        alphas = 1 - betas
        log_alphas = torch.log(alphas)
        for i in range(1, log_alphas.shape[0]):
            log_alphas[i] += log_alphas[i - 1]
        alpha_bars = log_alphas.exp()
        sigmas_flex = torch.sqrt(betas)
        sigmas_inflex = torch.zeros_like(sigmas_flex)
        for i in range(1, sigmas_flex.shape[0]):
            sigmas_inflex[i] = ((1 - alpha_bars[i - 1]) / (1 - alpha_bars[i])) * betas[i]
        self.num_steps = num_steps
        for name, t in (('betas', betas), ('alphas', alphas), ('alpha_bars', alpha_bars),
                        ('sigmas_flex', sigmas_flex), ('sigmas_inflex', torch.sqrt(sigmas_inflex))):
            self.register_buffer(name, t)

    def uniform_sample_t(self, batch_size):
        return torch.randint(1, self.num_steps + 1, (batch_size,)).tolist()

    def get_sigmas(self, t, flexibility=0):
        assert 0 <= flexibility <= 1
        return self.sigmas_flex[t] * flexibility + self.sigmas_inflex[t] * (1 - flexibility)


def respaced_timesteps(n_diff_steps, k):
    """The uniform 'trailing' respacing of a T-step schedule: round(i T / k) for i = k .. 1 (round half to even), a
    strictly decreasing list of k steps that starts at T.  k = T gives T, T - 1, ..., 1."""
    T, k = int(n_diff_steps), int(k)
    if not 1 <= k <= T:
        raise ValueError(f'k must be in [1, n_diff_steps = {T}], got {k}')
    return [round(Fraction(i * T, k)) for i in range(k, 0, -1)]


def respaced_coefficients(alpha_bars, timesteps, eta, target):
    """float64 (c0, c1, sigma) per visited step of a respaced schedule: x_s = c0 x_t + c1 out + sigma z with out the
    network output (x0_hat for target 'sample', eps_hat for 'noise'); s is the next entry (0 after the last, alpha_bars[0]
    = 1).  The engine plans the same coefficients on the host (include/msmd_b200.h, msmd_sample_schedule)."""
    ab = torch.as_tensor(alpha_bars).double().cpu()
    t = torch.tensor([int(v) for v in timesteps])
    s = torch.cat([t[1:], torch.zeros(1, dtype=t.dtype)])
    A = ab[t]
    B = torch.where(s > 0, ab[s], torch.ones_like(A))
    sigma = eta * torch.sqrt((1 - B) / (1 - A)) * torch.sqrt(torch.clamp(1 - A / B, min=0))
    r = torch.sqrt(torch.clamp(1 - B - sigma ** 2, min=0))
    if target == 'noise':
        c0 = torch.sqrt(B / A)
        c1 = r - torch.sqrt(B) * torch.sqrt(1 - A) / torch.sqrt(A)
    else:
        c0 = r / torch.sqrt(1 - A)
        c1 = torch.sqrt(B) - torch.sqrt(A) * c0
    return c0, c1, sigma


def dpmpp_2m_coefficients(alpha_bars, timesteps, eta, target, start=0, first=True):
    """float64 (c0, c1, c2, sigma, a, b) per step of DPM-Solver++(2M) on a respaced schedule, for a call that runs
    timesteps[start:]: x_s = c0 x_t + c1 out + c2 x0_p + sigma z with out the network output, x0_p the data prediction
    of the previous step and x0_t = a x_t + b out this step's (a = 0, b = 1 for target 'sample').  The first step is
    first order when ``first`` (no predecessor: a call without x0_prev), else its predecessor is timesteps[start - 1]
    (x0_prev); the step to s = 0 is first order.  A call of fewer steps uses a prefix of the rows.  The engine plans
    the same coefficients on the host (include/msmd_b200.h, msmd_sample_schedule)."""
    ab = torch.as_tensor(alpha_bars).double().cpu().tolist()
    ts = [int(v) for v in timesteps]
    if not first and start == 0:
        raise ValueError('first=False needs a predecessor: start must be > 0')
    lam = lambda A: math.log(math.sqrt(A) / math.sqrt(1 - A))
    rows = []
    for i in range(start, len(ts)):
        t, s = ts[i], (ts[i + 1] if i + 1 < len(ts) else 0)
        al_t, sg_t = math.sqrt(ab[t]), math.sqrt(1 - ab[t])
        k, M, sigma, w1, w2 = 0.0, 1.0, 0.0, 1.0, 0.0      # s = 0: x_0 = x0_t
        if s > 0:
            al_s, sg_s = math.sqrt(ab[s]), math.sqrt(1 - ab[s])
            h = lam(ab[s]) - lam(ab[t])
            k = sg_s / sg_t * math.exp(-eta * h)
            M = -al_s * math.expm1(-(1 + eta) * h)
            sigma = sg_s * math.sqrt(-math.expm1(-2 * eta * h))
            if i > start or not first:
                r = (lam(ab[t]) - lam(ab[ts[i - 1]])) / h
                w1, w2 = 1 + 0.5 / r, -0.5 / r
        a, b = (1 / al_t, -sg_t / al_t) if target == 'noise' else (0.0, 1.0)
        rows.append([k + M * w1 * a, M * w1 * b, M * w2, sigma, a, b])
    return tuple(torch.tensor(rows, dtype=torch.float64).T)


def hybrid_bounds(timesteps, w1, w2, tol, err16, err_main, k32=None):
    """Segment bounds (k32, k16) of the hybrid arithmetic on a visited-step list: steps with t <= k32 run fp32-grade
    (error 0), t <= k16 fp16 (err16), the others the main 16-bit arithmetic (err_main).  Step j carries
    w1[j] err(t_j) + w2[j] err(t_{j-1}): its own output's error and that of the previous step's output, which a
    multistep solver reuses.  k32 (unless given) is the smallest bound, 0 or a visited t, with every step within tol
    when k16 = T; then k16 is the smallest bound >= k32 that keeps every step within tol.  Feasibility is monotone in
    both bounds, so each is the largest of the per-step minima."""
    ts = [int(t) for t in timesteps]
    w1, w2 = [float(v) for v in w1], [float(v) for v in w2]

    def ok(j, b32, b16):
        e = lambda t: 0.0 if t <= b32 else (err16 if t <= b16 else err_main)
        return w1[j] * e(ts[j]) + (w2[j] * e(ts[j - 1]) if j else 0.0) <= tol

    prev = lambda j: ts[j - 1] if j else ts[j]
    if k32 is None:
        k32 = max(next((b for b in (0, ts[j]) if ok(j, b, ts[0])), prev(j)) for j in range(len(ts)))
    k16 = max(next((b for b in (k32, max(k32, ts[j])) if ok(j, k32, b)), max(k32, prev(j))) for j in range(len(ts)))
    return k32, k16


def _engine_cfg(net, n_diff_steps, target, max_seqs, precision='bf16'):
    if precision not in PRECISIONS:
        raise ValueError(f"precision must be one of {sorted(PRECISIONS)}, got {precision!r}")
    return dict(n_motions=net.n_motions, n_prev_motions=net.n_prev_motions, d_model=net.feature_dim,
                n_heads=net.n_heads, n_layers=net.n_layers, d_ff=net.mlp_ratio * net.feature_dim,
                d_style=net.style_feat_dim if net.use_style else 0, d_shape=net.shape_feat_dim,
                motion_dim=net.motion_feat_dim, n_basis=net.num_of_basis, n_diff_steps=n_diff_steps,
                use_indicator=int(bool(net.use_indicator)), align_mask_width=net.align_mask_width,
                target_noise=int(target == 'noise'), max_seqs=max_seqs, precision=PRECISIONS[precision])


def _check_alignment_mask(net):
    """The engine builds the cross-attention band from ``align_mask_width`` and never reads the bool
    ``alignment_mask`` buffer (only floating-point entries are packed).  A buffer that disagrees with the width, e.g. one
    overwritten by a checkpoint loaded with ``strict=True``, would be silently ignored, so it raises instead."""
    w = net.align_mask_width
    got = getattr(net, 'alignment_mask', None)
    if w <= 0:
        if got is not None:
            raise _lib.MsmdError(f'alignment_mask is set but align_mask_width={w} means no cross-attention mask')
        return
    n = net.n_prev_motions + net.n_motions
    want = torch.nn.functional.pad(enc_dec_mask(n, n, 1, w - 1, device='cpu'), (0, 0, 1, 0), value=False)
    if got is None or tuple(got.shape) != tuple(want.shape) or not torch.equal(got.detach().cpu().bool(), want):
        raise _lib.MsmdError(f'alignment_mask does not match align_mask_width={w}: the engine applies the band of the '
                             'width, so the module buffer must equal enc_dec_mask(n, n, 1, w-1) with an all-visible row 0')


class _EngineOwner:
    """Mixin: lazily creates / grows the CUDA engine and keeps its packed weights in sync with the module.

    ``precision`` picks the engine arithmetic.  The reference runs plain fp32 (no autocast), so the default is the
    mode that keeps EVERY sampling step within 1e-3 relative L2 of it:
      'hybrid' (default)  bf16 tensor-core steps while the posterior coefficient c1(t) damps their 6.5e-3 x0_hat
                          error below 1e-3, one-pass fp16 steps (same cost, error 8e-4) for the last ``fp16_last_steps``,
                          fp32-grade steps (3-pass fp16-split GEMMs, error 2e-6) for the last ``precise_last_steps``;
      'fp32'              every step fp32-grade (<= 1e-5);
      'bf16' / 'fp16'     explicit opt-in: one 16-bit arithmetic for every step (the last steps miss 1e-3 in bf16)."""
    precision = 'hybrid'
    precise_last_steps = 'auto'   # int, or 'auto' = MSMD.auto_steps(FP16_ERR_BOUND): steps the fp16 path could miss 1e-3 on
    fp16_last_steps = 'auto'      # int, or 'auto' = MSMD.auto_steps(BF16_ERR_BOUND)

    def _engine_state(self):
        raise NotImplementedError

    def check(self):
        """Synchronise and raise if an earlier fp32-grade call left the fp16 range of its operand split (the sampling
        call itself never synchronises; it poisons its output with NaN and reports at the next call)."""
        eng = getattr(self, '_eng', None)
        if eng is not None:
            eng.check()

    def _get_engine(self, n_seqs, device):
        cfg_fn, sd_fn = self._engine_state()
        eng = getattr(self, '_eng', None)
        if eng is None or eng.device != device or eng.cfg.max_seqs < n_seqs or eng.cfg.precision != cfg_fn(1)['precision']:
            cap = max(n_seqs, 0 if eng is None else eng.cfg.max_seqs)
            eng = DenoiserEngine(cfg_fn(cap), device)
            object.__setattr__(self, '_eng', eng)
        sd = sd_fn()
        key = tuple((k, v.data_ptr(), v._version) for k, v in sd.items())
        if eng.weights_key != key:
            _check_alignment_mask(getattr(self, 'denoising_net', self))   # MSMD holds the network, which owns the buffer
            eng.load_state_dict(sd)
            eng.weights_key = key
        return eng


class DenoisingNetwork_MSMD(nn.Module, _EngineOwner):
    """model.py:820-996.  Parameter container + forward through the engine."""

    def __init__(self, args, device='cuda', motion_feat_dim=50, use_head_alpha=True, regularize_alpha="None"):
        super().__init__()
        self.regularize_alpha = regularize_alpha
        self.use_head_alpha = use_head_alpha
        self.num_of_basis = int(args.num_of_basis)
        self.use_style = args.style_enc_ckpt is not None or not args.style_enc_model_style == "diffposetalk"
        self.motion_feat_dim = motion_feat_dim
        if (args.dataset_type[:9] == "HDTF_TFHP" or args.dataset_type == 'flame_mead_ravdess') and motion_feat_dim == 50:
            if args.rot_repr != 'aa':
                raise ValueError(f'Unknown rotation representation {args.rot_repr}!')
            self.motion_feat_dim += 1 if args.no_head_pose else 4
        self.shape_feat_dim = 100
        self.style_feat_dim = args.d_style if self.use_style else 0
        self.person_feat_dim = self.shape_feat_dim + self.style_feat_dim
        self.use_indicator = args.use_indicator
        self.architecture = args.architecture
        self.feature_dim, self.n_heads, self.n_layers = args.feature_dim, args.n_heads, args.n_layers
        self.mlp_ratio, self.align_mask_width = args.mlp_ratio, args.align_mask_width
        self.use_learnable_pe = not args.no_use_learnable_pe
        self.n_prev_motions, self.n_motions = args.n_prev_motions, args.n_motions
        self._n_diff_steps = args.n_diff_steps
        if self.architecture != 'decoder':
            raise ValueError(f'Unknown architecture: {self.architecture}')
        if not self.use_learnable_pe:
            raise _lib.MsmdError('msmd_b200: only the learnable positional encoding (no_use_learnable_pe=False) is built')
        if use_head_alpha or regularize_alpha == "sigmoid":
            raise _lib.MsmdError('msmd_b200: use_head_alpha / sigmoid alphas are not built '
                                 '(get_diffusion_model always passes use_head_alpha=False, model.py:17)')
        d = self.feature_dim
        self.TE = PositionalEncoding(d, max_len=args.n_diff_steps + 1)
        self.diff_step_map = nn.Sequential(nn.Linear(d, d), nn.GELU(), nn.Linear(d, d))
        self.PE = nn.Parameter(torch.randn(1, 1 + self.n_prev_motions + self.n_motions, d))
        self.person_proj = nn.Linear(self.person_feat_dim, d)
        self.feature_proj = nn.Linear(self.motion_feat_dim + (1 if self.use_indicator else 0), d)
        layer = nn.TransformerDecoderLayer(d_model=d, nhead=self.n_heads, dim_feedforward=self.mlp_ratio * d,
                                           activation='gelu', batch_first=True)
        self.transformer = nn.TransformerDecoder(layer, num_layers=self.n_layers)   # parameter holder only
        if self.align_mask_width > 0:
            n = self.n_prev_motions + self.n_motions
            mask = enc_dec_mask(n, n, 1, self.align_mask_width - 1, device='cpu')
            self.register_buffer('alignment_mask', torch.nn.functional.pad(mask, (0, 0, 1, 0), value=False))
        else:
            self.alignment_mask = None
        self.static_feature_mapping = nn.ModuleList(
            nn.Sequential(nn.Linear(args.d_style, d), nn.GELU(), nn.Linear(d, self.motion_feat_dim))
            for _ in range(self.num_of_basis))
        self.motion_dec = nn.Sequential(nn.Linear(d, d // 2), nn.GELU(),
                                        nn.Linear(d // 2, self.motion_feat_dim + self.num_of_basis))
        self.to(device)

    @property
    def device(self):
        return next(self.parameters()).device

    def _engine_state(self):
        # standalone module use: the tables only feed the sampler.  Built once: a fresh schedule per call changed the
        # weights key (new data_ptrs) and forced a full weight re-pack on every forward.
        sched = self.__dict__.get('_sched')
        if sched is None:
            sched = DiffusionSchedule(self._n_diff_steps, 'cosine')
            self.__dict__['_sched'] = sched
        def sd():
            out = {'denoising_net.' + k: v for k, v in self.state_dict().items()}
            out.update({'diffusion_sched.' + k: v for k, v in sched.state_dict().items()})
            return out
        return (lambda cap: _engine_cfg(self, self._n_diff_steps, 'sample', cap, self.precision)), sd

    @torch.no_grad()
    def forward(self, motion_feat, audio_feat, person_feat, static_style_feat, prev_motion_feat, prev_audio_feat,
                step, indicator=None, keep_separate=False, precise=None):
        """model.py:914-996.  ``keep_separate`` returns (dynamic_features [N,Lp+L,dm], static_features [N,Lp+L,nb,dm],
        alphas [N,Lp+L,nb]) like the reference (:972-973).  ``precise`` (extra): None = the most accurate arithmetic
        the engine holds (fp32-grade unless precision is 'bf16'/'fp16'), True/False, or 'bf16' / 'fp16' / 'fp32'."""
        if self.use_indicator and indicator is None:
            raise ValueError('indicator is required when use_indicator is set')
        N = motion_feat.shape[0]
        eng = self._get_engine(N, motion_feat.device)
        eng.window_begin(audio_feat, person_feat.reshape(N, -1), static_style_feat.reshape(N, -1), prev_motion_feat,
                         prev_audio_feat, indicator, NX=N, E=1)
        steps = torch.as_tensor(step).reshape(-1).expand(N)
        if keep_separate:
            return eng.denoise_parts(motion_feat, steps, precise)
        return eng.denoise(motion_feat, steps, precise)


class MSMD(nn.Module, _EngineOwner):
    """model.py:73-818 (inference surface: sample, extract_audio_feature)."""

    def __init__(self, args, device='cuda', vae_style=False, conditioned=True, denoisingnset_version=1,
                 use_head_alpha=True, regularize_alpha="None", audio_encoder=None):
        super().__init__()
        self.target = args.target
        self.regularize_alpha = regularize_alpha
        self.architecture = args.architecture
        self.use_style = (args.style_enc_ckpt is not None) or vae_style
        self.conditioned = conditioned
        self.motion_feat_dim = 67
        self.use_head_alpha = use_head_alpha
        self.fps, self.n_motions, self.n_prev_motions = args.fps, args.n_motions, args.n_prev_motions
        if self.use_style:
            self.style_feat_dim = args.d_style
        self.audio_model = args.audio_model
        if self.audio_model not in ('wav2vec2', 'hubert'):
            raise ValueError(f'Unknown audio model {self.audio_model}!')
        if audio_encoder is not None:
            self.audio_encoder = audio_encoder
        else:
            from .utils import hubert as _hub, wav2vec2 as _w2v
            self.audio_encoder = (_hub.HubertModel if self.audio_model == 'hubert' else _w2v.Wav2Vec2Model).from_pretrained(
                'facebook/hubert-base-ls960' if self.audio_model == 'hubert' else 'facebook/wav2vec2-base-960h')
        if args.architecture != 'decoder':
            raise ValueError(f'Unknown architecture {args.architecture}!')
        self.audio_feature_map = nn.Linear(768, args.feature_dim)
        self.start_audio_feat = nn.Parameter(torch.randn(1, self.n_prev_motions, args.feature_dim))
        self.start_motion_feat = nn.Parameter(torch.randn(1, self.n_prev_motions, self.motion_feat_dim))
        self.denoising_net = DenoisingNetwork_MSMD(args, device, motion_feat_dim=self.motion_feat_dim,
                                                   use_head_alpha=self.use_head_alpha,
                                                   regularize_alpha=self.regularize_alpha)
        self.diffusion_sched = DiffusionSchedule(args.n_diff_steps, args.diff_schedule)
        self.cfg_mode = args.cfg_mode
        conds = args.guiding_conditions.split(',') if args.guiding_conditions else []
        self.guiding_conditions = [c for c in conds if c in ['style', 'audio']]
        if 'style' in self.guiding_conditions:
            if not self.use_style:
                raise ValueError('Cannot use style guiding without enabling it!')
            self.null_style_feat = nn.Parameter(torch.randn(1, 1, self.style_feat_dim))
        if 'audio' in self.guiding_conditions:
            self.null_audio_feat = nn.Parameter(torch.randn(1, 1, args.feature_dim))
        self.to(device)

    @property
    def device(self):
        return next(self.parameters()).device

    def forward(self, *a, **k):
        raise _lib.MsmdError('msmd_b200 implements the inference path only; MSMD.forward (training noising / '
                             'CFG dropout, model.py:146-248) is out of scope')

    def _engine_state(self):
        net = self.denoising_net
        def sd():
            out = {'denoising_net.' + k: v for k, v in net.state_dict().items()}
            out.update({'diffusion_sched.' + k: v for k, v in self.diffusion_sched.state_dict().items()})
            return out
        return (lambda cap: _engine_cfg(net, self.diffusion_sched.num_steps, self.target, cap, self.precision)), sd

    # x0_hat relative-L2 error bounds of the 16-bit paths vs the fp32 reference, = measured x a safety margin
    # (tests/test_denoiser_gpu.py asserts the measured values stay below them): bf16 6.5e-3 x 1.5, fp16 8e-4 x 2.5.
    BF16_ERR_BOUND = 1.0e-2
    FP16_ERR_BOUND = 2.0e-3

    def _output_weights(self, timesteps, eta, solver):
        """Per visited step: |coefficient| of this step's network output and of the previous step's output."""
        ab = self.diffusion_sched.alpha_bars
        if solver == 'dpmpp_2m':
            _, c1, c2, _, _, b = dpmpp_2m_coefficients(ab, timesteps, eta, self.target)
            return c1.abs().tolist(), [0.0] + (c2[1:] * b[:-1]).abs().tolist()
        _, c1, _ = respaced_coefficients(ab, timesteps, eta, self.target)
        return c1.abs().tolist(), [0.0] * len(c1)

    def auto_steps(self, err, tol=1e-3, timesteps=None, eta=None, solver='ddim'):
        """Number of final sampling steps on which a network-output error of ``err`` could exceed ``tol`` in x_{t-1}:
        x_{t-1} = c0 x_t + c1(t) x0_hat + sigma z carries the error scaled by c1(t), which decreases with t
        (c1(1) = 1, c1(2) = 0.52, c1(16) = 0.10 for the 500-step cosine schedule).  On a respaced schedule
        (``timesteps``, ``eta``, ``solver``): the smallest bound, 0 or a visited t, such that running the steps above
        it with error ``err`` keeps every step within tol (hybrid_bounds); for DDIM, the largest visited t whose
        |output coefficient| x err exceeds tol."""
        sch = self.diffusion_sched
        if timesteps is not None:
            w1, w2 = self._output_weights(timesteps, float(eta or 0.0), solver)
            return hybrid_bounds(timesteps, w1, w2, tol, err, err)[0]
        a, ab = sch.alphas.double().cpu(), sch.alpha_bars.double().cpu()
        t = torch.arange(1, sch.num_steps + 1)
        if self.target == 'noise':
            c1 = (1 - a[t]) / torch.sqrt(1 - ab[t]) / torch.sqrt(a[t])
        else:
            c1 = (1 - a[t]) * torch.sqrt(ab[t - 1]) / (1 - ab[t])
        over = torch.nonzero(c1 * err > tol)
        return int(over.max()) + 1 if len(over) else 0

    def auto_precise_steps(self, tol=1e-3):
        return self.auto_steps(self.FP16_ERR_BOUND, tol)

    def _precise_steps(self, override=None, timesteps=None, eta=None, solver='ddim'):
        """(fp32-grade last steps, fp16 last steps) of the hybrid schedule; (0, 0) for the single-arithmetic engines.
        Both are bounds in t: visited steps with t <= bound run the more precise arithmetic.  On a respaced schedule
        both come from hybrid_bounds."""
        if self.precision != 'hybrid':
            return 0
        k = self.precise_last_steps if override is None else override
        return self.auto_steps(self.FP16_ERR_BOUND, timesteps=timesteps, eta=eta, solver=solver) if k == 'auto' else int(k)

    def _fp16_steps(self, override=None, timesteps=None, eta=None, solver='ddim', precise_override=None):
        if self.precision != 'hybrid':
            return 0
        k = self.fp16_last_steps if override is None else override
        if k != 'auto':
            return int(k)
        if timesteps is None:
            return self.auto_steps(self.BF16_ERR_BOUND)
        w1, w2 = self._output_weights(timesteps, float(eta or 0.0), solver)
        k32 = self._precise_steps(precise_override, timesteps, eta, solver)
        return hybrid_bounds(timesteps, w1, w2, 1e-3, self.FP16_ERR_BOUND, self.BF16_ERR_BOUND, k32=k32)[1]

    @torch.no_grad()
    def extract_audio_feature(self, audio, frame_num=None):
        """model.py:250-264: [N, samples] -> [N, frame_num, feature_dim], all inside the CUDA audio encoder."""
        frame_num = frame_num or self.n_motions
        return self.audio_encoder.extract(audio, self.fps, frame_num, self.audio_feature_map)

    @torch.no_grad()
    def sample(self, audio_or_feat, shape_feat, style_feat=None, prev_motion_feat=None, prev_audio_feat=None,
               motion_at_T=None, indicator=None, cfg_mode=None, cfg_cond=None, cfg_scale=1.15, flexibility=0,
               dynamic_threshold=None, ret_traj=False, noise=None, n_steps=None, t_start=None, _separate=False,
               precise_last_steps=None, fp16_last_steps=None, noise_seed=None, clip_offset=0, noise_keys=None,
               timesteps=None, eta=None, solver='ddim', x0_prev=None):
        """model.py:282-440.  Extra keyword arguments (not in the reference): ``noise`` = externally supplied
        z tensor [T+1, N, L, 67] indexed by step t (default: in-kernel Philox seeded from torch's generator);
        ``t_start`` / ``n_steps`` = start at step t_start (motion_at_T is then x_{t_start}) and run n steps
        (teacher-forced parity tests); ``precise_last_steps`` / ``fp16_last_steps`` = with ``self.precision == 'hybrid'``,
        run the steps t <= precise_last_steps in fp32-grade and precise_last_steps < t <= fp16_last_steps in one-pass
        fp16 arithmetic (defaults: the attributes of the same names, 'auto'); ``noise_seed`` / ``clip_offset`` = key of the
        in-kernel Philox step noise (used when ``noise`` is None): clip n draws the stream of global clip clip_offset + n
        under ``noise_seed`` (default: a seed drawn from torch's generator), so clip-sharded runs reproduce the
        single-GPU codes (SURVEY 8(e)); ``noise_keys`` = int64 [N, 2] of (seed, global clip id) per clip, instead of
        ``noise_seed`` / ``clip_offset``, so one call can carry clips of different windows (inference.infer_coeffs_queue);
        ``timesteps`` / ``eta`` = sample on a respaced (DDIM) schedule: a strictly decreasing list of visited steps in
        [1, T] (e.g. respaced_timesteps(T, 50)) and eta in [0, 1] (default 0, deterministic), with ``flexibility`` 0.
        ``t_start`` must then be an entry of the list and ``n_steps`` counts list entries; ``ret_traj`` returns x_t
        over the visited t and 0.  ``solver`` = 'ddim' or 'dpmpp_2m' (DPM-Solver++(2M), second order with one network
        evaluation per step; its SDE variant for eta > 0), which needs ``timesteps``; ``x0_prev`` = [N, L, 67] CUDA
        tensor, the data prediction of the list entry before ``t_start`` (2M only), so a call that starts mid-list takes
        its first step at second order (without it the first step of a call is first order)."""
        N = audio_or_feat.shape[0]
        if solver not in ('ddim', 'dpmpp_2m'):
            raise ValueError(f"solver must be 'ddim' or 'dpmpp_2m', got {solver!r}")
        if x0_prev is not None:
            if solver != 'dpmpp_2m':
                raise ValueError("x0_prev applies to solver='dpmpp_2m'")
            if not isinstance(x0_prev, torch.Tensor) or not x0_prev.is_cuda or \
                    tuple(x0_prev.shape) != (N, self.n_motions, self.motion_feat_dim):
                raise ValueError(f'x0_prev must be a CUDA tensor [N, L, d] = [{N}, {self.n_motions}, '
                                 f'{self.motion_feat_dim}], got {tuple(getattr(x0_prev, "shape", ()))}')
        if timesteps is None:
            if eta is not None:
                raise ValueError('eta applies to a respaced schedule: pass timesteps too')
            if solver != 'ddim':
                raise ValueError("solver='dpmpp_2m' needs a respaced schedule: pass timesteps")
        else:
            if isinstance(timesteps, torch.Tensor):
                timesteps = timesteps.reshape(-1).tolist()
            timesteps = [int(t) for t in timesteps]
            T_all = self.diffusion_sched.num_steps
            if not timesteps or any(not 1 <= t <= T_all for t in timesteps) or \
                    any(b >= a for a, b in zip(timesteps, timesteps[1:])):
                raise ValueError(f'timesteps must be a non-empty, strictly decreasing list in [1, {T_all}]')
            eta = 0.0 if eta is None else float(eta)
            if not 0.0 <= eta <= 1.0:
                raise ValueError(f'eta must be in [0, 1], got {eta}')
            if flexibility != 0:
                raise ValueError('flexibility has no meaning on a respaced schedule: it must be 0 with timesteps')
            if t_start is not None and t_start not in timesteps:
                raise ValueError(f't_start {t_start} is not an entry of timesteps')
            if x0_prev is not None and (t_start or timesteps[0]) == timesteps[0]:
                raise ValueError("x0_prev needs a predecessor: t_start must not be timesteps' first entry")
        if noise_keys is not None:
            if not isinstance(noise_keys, torch.Tensor) or noise_keys.dtype != torch.int64 or \
                    tuple(noise_keys.shape) != (N, 2):
                raise ValueError(f'noise_keys must be an int64 tensor [N, 2] = [{N}, 2], got '
                                 f'{getattr(noise_keys, "dtype", type(noise_keys))} {tuple(getattr(noise_keys, "shape", ()))}')
            if noise is not None or noise_seed is not None or clip_offset != 0:
                raise ValueError('noise_keys replace noise_seed / clip_offset and exclude an external noise tensor')
        dev = self.device
        cfg_mode = self.cfg_mode if cfg_mode is None else cfg_mode
        cfg_cond = self.guiding_conditions if cfg_cond is None else cfg_cond
        cfg_cond = [c for c in cfg_cond if c in ['audio', 'style']]
        if not isinstance(cfg_scale, list):
            cfg_scale = [cfg_scale] * len(cfg_cond)
        if len(cfg_cond) > 0:
            cfg_cond, cfg_scale = zip(*sorted(zip(cfg_cond, cfg_scale), key=lambda x: ['audio', 'style'].index(x[0])))
        else:
            cfg_cond, cfg_scale = [], []
        if cfg_mode not in ('independent', 'incremental'):
            raise NotImplementedError(f'Unknown cfg_mode {cfg_mode}')
        if 'style' in cfg_cond:
            assert self.use_style and style_feat is not None
        if self.use_style:
            if style_feat is None:
                style_feat = self.null_style_feat.expand(N, -1, -1)
        else:
            assert style_feat is None, 'This model does not support style feature input!'
        if audio_or_feat.ndim == 2:
            assert audio_or_feat.shape[1] == 16000 * self.n_motions / self.fps, \
                f'Incorrect audio length {audio_or_feat.shape[1]}'
            audio_feat = self.extract_audio_feature(audio_or_feat)
        elif audio_or_feat.ndim == 3:
            assert audio_or_feat.shape[1] == self.n_motions, f'Incorrect audio feature length {audio_or_feat.shape[1]}'
            audio_feat = audio_or_feat
        else:
            raise ValueError(f'Incorrect audio input shape {audio_or_feat.shape}')
        if shape_feat.ndim == 2:
            shape_feat = shape_feat.unsqueeze(1)
        if style_feat is not None and style_feat.ndim == 2:
            style_feat = style_feat.unsqueeze(1)
        if prev_motion_feat is None:
            prev_motion_feat = self.start_motion_feat.expand(N, -1, -1)
        if prev_audio_feat is None:
            prev_audio_feat = self.start_audio_feat.expand(N, -1, -1)
        if motion_at_T is None:
            motion_at_T = torch.randn((N, self.n_motions, self.motion_feat_dim)).to(dev)   # drawn on CPU (model.py:337)

        # conditioning of the E = 1 + len(cfg_cond) guidance entries (model.py:339-374)
        a_null = self.null_audio_feat.expand(N, self.n_motions, -1) if 'audio' in cfg_cond else audio_feat
        if 'style' in cfg_cond:
            p_null = torch.cat([shape_feat, self.null_style_feat.expand(N, -1, -1)], dim=-1)
        else:
            p_null = torch.cat([shape_feat, style_feat], dim=-1) if self.use_style else shape_feat
        audio_in, person_in = [a_null], [p_null]
        for cond in cfg_cond:
            if cond == 'audio':
                audio_in.append(audio_feat)
                person_in.append(p_null)
            else:
                audio_in.append(a_null if cfg_mode == 'independent' else audio_feat)
                person_in.append(torch.cat([shape_feat, style_feat], dim=-1))
        E = len(audio_in)
        rep = lambda t: torch.cat([t] * E, dim=0)
        eng = self._get_engine(N * E, dev)
        eng.window_begin(torch.cat(audio_in, 0), torch.cat(person_in, 0).reshape(N * E, -1),
                         rep(style_feat).reshape(N * E, -1), rep(prev_motion_feat), rep(prev_audio_feat),
                         rep(indicator) if indicator is not None else None, NX=N, E=E)
        if noise is not None or noise_keys is not None:
            seed = 0
        elif noise_seed is not None:
            seed = int(noise_seed)
        else:
            seed = int(torch.randint(0, 2 ** 62, (1,)).item())
        s0 = float(cfg_scale[0]) if E > 1 else 0.0
        s1 = float(cfg_scale[1]) if E > 2 else 0.0
        T = t_start or (timesteps[0] if timesteps is not None else self.diffusion_sched.num_steps)
        visited = None
        if timesteps is not None:
            visited = timesteps[timesteps.index(T):]
            n_steps = n_steps or len(visited)
            visited = visited[:n_steps]
        res = eng.sample_window(motion_at_T, noise, seed, cfg_mode == 'independent', s0, s1, flexibility,
                                t_start=T, n_steps=n_steps, want_traj=ret_traj, dynamic_threshold=dynamic_threshold,
                                separate=_separate,
                                precise_last_steps=self._precise_steps(precise_last_steps, timesteps, eta, solver),
                                fp16_last_steps=self._fp16_steps(fp16_last_steps, timesteps, eta, solver,
                                                                 precise_last_steps),
                                noise_clip_offset=clip_offset, noise_keys=noise_keys, timesteps=timesteps, eta=eta,
                                solver=solver, x0_prev=x0_prev)
        x0, traj = res[0], res[1]
        if _separate and not ret_traj:
            return x0, motion_at_T, audio_feat, res[2]
        if ret_traj and visited is not None:
            # x_s at each visited step's successor s (the list's next entry, 0 after the last)
            nxt = timesteps[timesteps.index(visited[-1]) + 1] if visited[-1] != timesteps[-1] else 0
            out = {T: motion_at_T.cpu()}
            out.update({t: traj[t].cpu() for t in visited[1:]})
            out[nxt] = traj[nxt]
            return out, motion_at_T, audio_feat
        if ret_traj:
            last = T - (n_steps or T)
            out = {T: motion_at_T.cpu()}
            out.update({t: traj[t].cpu() for t in range(T - 1, last, -1)})
            out[last] = traj[last]
            return out, motion_at_T, audio_feat
        return x0, motion_at_T, audio_feat


def _sample_separate(self, audio_or_feat, shape_feat, style_feat=None, prev_motion_feat=None, prev_audio_feat=None,
                     motion_at_T=None, indicator=None, cfg_mode=None, cfg_cond=None, cfg_scale=1.15, flexibility=0,
                     dynamic_threshold=None, ret_traj=False, alpah_t_modification=None, return_all_alpha=False,
                     noise=None, n_steps=None, timesteps=None, eta=None, solver='ddim'):
    """model.py:442-651.  Same loop as ``sample`` plus the decomposition outputs:
    (x0, x_T, audio_feat, target_dynamic, cumulative_static, alpha) with alpha = all steps concatenated along
    dim 0 (return_all_alpha) or the last step's [N, L, n_basis].  ``alpah_t_modification`` (a Python callback on
    the alphas of every step) cannot run inside the fused loop and must be None.  ``timesteps`` / ``eta``: a respaced
    schedule as in ``MSMD.sample``; alpha then has one entry per visited step.  Only ``solver='ddim'``: the
    cumulative static part of DPM-Solver++(2M) would need a second history buffer."""
    if solver != 'ddim':
        raise ValueError(f"sample_separate supports solver='ddim' only, got {solver!r}")
    if alpah_t_modification is not None:
        raise _lib.MsmdError('msmd_b200: alpah_t_modification callbacks are not supported by the fused sampler')
    out = self.sample(audio_or_feat, shape_feat, style_feat, prev_motion_feat, prev_audio_feat, motion_at_T, indicator,
                      cfg_mode, cfg_cond, cfg_scale, flexibility, dynamic_threshold, ret_traj, noise=noise,
                      n_steps=n_steps, _separate=True, timesteps=timesteps, eta=eta)
    if ret_traj:
        return out
    x0, x_T, audio_feat, (tgt_dyn, cum_static, alpha_traj) = out
    alpha = alpha_traj.reshape(-1, *alpha_traj.shape[2:]) if return_all_alpha else alpha_traj[-1]
    return x0, x_T, audio_feat, tgt_dyn, cum_static, alpha


MSMD.sample_separate = torch.no_grad()(_sample_separate)
