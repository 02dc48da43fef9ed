"""Drop-in for the hot-path driver of /root/reference/inference.py: ``infer_coeffs`` (inference.py:34-75).

Same signature and windowing semantics: the audio encoder sees the whole zero-padded clip once, windows
of ``n_motions`` frames are sampled sequentially, each conditioned on the previous window's last
``n_prev_motions`` frames of motion and of INPUT audio features, every window re-uses window 0's x_T
(inference.py:57-69, SURVEY App. C-5), and the padded tail is trimmed.

``infer_coeffs_batched`` is the same loop over a batch of independent clips (the reference handles one
clip per call; clips never interact, so they are simply stacked along the batch dimension).

``infer_coeffs_queue`` / ``infer_coeffs_many`` sample clips of different lengths with a clip queue: every sampler call
keeps up to ``max_clips`` clips in flight, whatever window each of them is on, and each clip's step noise is keyed by
its own (seed + window, global clip id).
"""
import math

import torch
import torch.nn.functional as F


@torch.no_grad()
def infer_coeffs_batched(model, args, audio_feat, shape_coef, style_feats=None, clip_len=None, cfg_mode=None,
                         cfg_cond=None, cfg_scale=1.15, dynamic_threshold=None, x_T=None, noise=None, noise_seed=None,
                         clip_offset=0, timesteps=None, eta=None, solver='ddim'):
    """audio_feat [N, n_sub*n_motions, d] (already extracted); shape_coef [N,1,100] or [N,100];
    style_feats [N,d_style] (or a list per window); clip_len = frames to keep (<= n_sub*n_motions).
    x_T [N,n_motions,67] / noise ([T+1,N,L,67] or a list per window) are optional fixed inputs; without ``noise`` the
    step noise is the in-kernel Philox stream keyed by (noise_seed + window, global clip id = clip_offset + n), so the
    codes of a clip do not depend on which batch / GPU it was sampled in.  ``timesteps`` / ``eta`` / ``solver``: sample
    every window on a respaced schedule (MSMD.sample).
    Returns [N, clip_len, 67]."""
    N, total = audio_feat.shape[:2]
    L = args.n_motions
    assert total % L == 0, f'audio feature length {total} is not a multiple of n_motions={L}'
    n_sub = total // L
    clip_len = total if clip_len is None else clip_len
    n_padding_frames = total - clip_len
    coef_list = []
    prev_motion_feat = prev_audio_feat = None
    noise_T = x_T
    for i in range(n_sub):
        indicator = torch.ones((N, L), device=audio_feat.device) if args.use_indicator else None
        if indicator is not None and i == n_sub - 1 and n_padding_frames > 0:
            indicator[:, -n_padding_frames:] = 0
        audio_in = audio_feat[:, i * L:(i + 1) * L]
        style_feat = style_feats[i] if isinstance(style_feats, list) else style_feats
        z = noise[i] if isinstance(noise, list) else noise
        motion_feat, noise_T, used_audio = model.sample(
            audio_in, shape_coef, style_feat, prev_motion_feat, prev_audio_feat, noise_T, indicator=indicator,
            cfg_mode=cfg_mode, cfg_cond=cfg_cond, cfg_scale=cfg_scale, dynamic_threshold=dynamic_threshold, noise=z,
            noise_seed=None if noise_seed is None else int(noise_seed) + i, clip_offset=clip_offset, timesteps=timesteps,
            eta=eta, solver=solver)
        prev_motion_feat = motion_feat[:, -args.n_prev_motions:].clone()
        prev_audio_feat = used_audio[:, -args.n_prev_motions:]
        if i == n_sub - 1 and n_padding_frames > 0:
            motion_feat = motion_feat[:, :-n_padding_frames]
        coef_list.append(motion_feat)
    return torch.cat(coef_list, dim=1)


def plan_clip(n_samples, args, audio_unit):
    """Windowing of one clip of ``n_samples`` 16 kHz samples (inference.py:39-45): (n_subdivision, samples after zero
    padding, clip_len = frames kept).  The clip is padded up to n_subdivision windows of audio, never truncated."""
    clip_len = int(n_samples / 16000 * args.fps)
    n_audio_samples = round(audio_unit * args.n_motions)
    n_subdivision = 1 if clip_len <= args.n_motions else math.ceil(clip_len / args.n_motions)
    n_padding_audio_samples = n_audio_samples * n_subdivision - n_samples
    n_padding_frames = math.ceil(n_padding_audio_samples / audio_unit)
    padded = n_samples + max(n_padding_audio_samples, 0)
    return n_subdivision, padded, args.n_motions * n_subdivision - max(n_padding_frames, 0)


@torch.no_grad()
def infer_coeffs(model, args, audio, shape_coef, audio_unit, style_feats=None, n_repetitions: int = 1, cfg_mode=None,
                 cfg_cond=None, cfg_scale: float = 1.15, include_shape: bool = False, dynamic_threshold=(0, 1, 4),
                 timesteps=None, eta=None, solver='ddim'):
    """inference.py:34-75 (one clip, 1-D 16 kHz audio).  ``timesteps`` / ``eta`` / ``solver``: a respaced schedule
    (MSMD.sample)."""
    n_subdivision, padded, clip_len = plan_clip(len(audio), args, audio_unit)
    if padded > len(audio):
        audio = F.pad(audio, (0, padded - len(audio)), value=0)
    audio_feat = model.extract_audio_feature(audio.unsqueeze(0), args.n_motions * n_subdivision)
    rep = lambda t: t if t is None else t.expand(n_repetitions, *t.shape[1:])
    style = [rep(s) for s in style_feats] if isinstance(style_feats, list) else rep(style_feats)
    return infer_coeffs_batched(model, args, audio_feat.expand(n_repetitions, -1, -1), rep(shape_coef), style,
                                clip_len=clip_len, cfg_mode=cfg_mode, cfg_cond=cfg_cond,
                                cfg_scale=cfg_scale, dynamic_threshold=dynamic_threshold, timesteps=timesteps, eta=eta,
                                solver=solver)


def queue_schedule(n_windows, max_clips):
    """Sampler calls of the clip queue: a list of calls, each a list of (clip, window) in slot order.  At most
    ``max_clips`` clips are in flight; clips are admitted in order; a clip that has run its last window hands its
    slot to the next queued clip at the next window boundary (slots left without a clip close up)."""
    if max_clips < 1:
        raise ValueError(f'max_clips must be >= 1, got {max_clips}')
    if any(n < 1 for n in n_windows):
        raise ValueError('every clip needs at least one window')
    slots, calls, nxt = [], [], 0
    while nxt < len(n_windows) and len(slots) < max_clips:
        slots.append([nxt, 0])
        nxt += 1
    while slots:
        calls.append([(k, w) for k, w in slots])
        kept = []
        for k, w in slots:
            if w + 1 < n_windows[k]:
                kept.append([k, w + 1])
            elif nxt < len(n_windows):
                kept.append([nxt, 0])
                nxt += 1
        slots = kept
    return calls


@torch.no_grad()
def infer_coeffs_queue(model, args, audio_feats, shape_coefs, style_feats, clip_lens, x_T, max_clips=64, clip_ids=None,
                       noise_seed=0, cfg_mode=None, cfg_cond=None, cfg_scale=1.15, dynamic_threshold=None, timesteps=None,
                       eta=None, solver='ddim'):
    """``infer_coeffs_batched`` over clips of different lengths, keeping up to ``max_clips`` clips in every sampler call.

    Per clip k: audio_feats[k] [n_sub_k * n_motions, d] (already extracted), shape_coefs[k] [100] / [1, 100],
    style_feats[k] [d_style] (or style_feats None), clip_lens[k] frames to keep, x_T[k] [n_motions, 67] (re-used by every
    window, like infer_coeffs_batched).  One call mixes clips that are on different windows (queue_schedule); the step
    noise of clip k's window w is keyed by (noise_seed + w, clip_ids[k]) (default clip_ids: 0..K-1), so clip k's codes
    are those of infer_coeffs_batched on that clip alone with noise_seed and clip_offset = clip_ids[k].
    The schedule depends on the lengths only: nothing is read back from the device between windows.  ``timesteps`` /
    ``eta`` / ``solver``: every call samples on this one respaced schedule (the clips of a call share the step index;
    every call runs a whole window, so a 2M call starts first order).
    Returns (codes [K, max_k clip_lens[k], 67], zero beyond each clip's length; lengths [K] int64)."""
    K = len(audio_feats)
    if K == 0:
        raise ValueError('infer_coeffs_queue: no clips')
    clip_ids = list(range(K)) if clip_ids is None else [int(i) for i in clip_ids]
    others = dict(shape_coefs=shape_coefs, clip_lens=clip_lens, x_T=x_T, clip_ids=clip_ids)
    if style_feats is not None:
        others['style_feats'] = style_feats
    bad = {k: len(v) for k, v in others.items() if len(v) != K}
    if bad:
        raise ValueError(f'infer_coeffs_queue: {K} audio feature tensors but {bad}')
    L, Lp = args.n_motions, args.n_prev_motions
    n_sub = []
    for k, (f, n) in enumerate(zip(audio_feats, clip_lens)):
        if f.ndim != 2 or f.shape[0] % L or f.shape[0] == 0:
            raise ValueError(f'clip {k}: audio features must be [n_sub * {L}, d], got {tuple(f.shape)}')
        if not (f.shape[0] - L <= int(n) <= f.shape[0]):
            raise ValueError(f'clip {k}: clip_len {int(n)} outside its last window ({f.shape[0] - L}, {f.shape[0]}]')
        n_sub.append(f.shape[0] // L)
    calls = queue_schedule(n_sub, max_clips)
    dev = model.device
    W = max(n_sub)
    # the small per-clip inputs are stacked once and each call gathers its rows with index tensors planned (and uploaded)
    # up front; the audio features stay in the caller's per-clip tensors (a dense [K, W*L, d] copy would grow with
    # K x the longest clip) and each call stacks its windows' slices (views) with one copy
    feats = [f.to(dev) for f in audio_feats]
    start_audio = model.start_audio_feat.detach()[0]
    shape = torch.stack([s.reshape(1, -1) for s in shape_coefs]).to(dev)
    style = None if style_feats is None else torch.stack([s.reshape(-1) for s in style_feats]).to(dev)
    xT = torch.stack([x.reshape(L, -1) for x in x_T]).to(dev)
    prev_motion = model.start_motion_feat.detach().expand(K, -1, -1).clone()
    codes = torch.zeros((K, W * L, xT.shape[-1]), device=dev)
    plan = []                                    # per call: clip, window, valid frames, seed, global clip id
    for call in calls:
        for k, w in call:
            valid = int(clip_lens[k]) - w * L if w == n_sub[k] - 1 else L
            plan.append((k, w, valid, int(noise_seed) + w, clip_ids[k]))
    plan = torch.tensor(plan, dtype=torch.int64)
    plan = (plan.pin_memory() if dev.type == 'cuda' else plan).to(dev, non_blocking=True)
    frames = torch.arange(L, device=dev)
    pos = 0
    for call in calls:
        n = len(call)
        p = plan[pos:pos + n]
        pos += n
        idx, win = p[:, 0], p[:, 1]
        rows = win[:, None] * L + frames                                  # [n, L] frames of this window
        audio_in = torch.stack([feats[k][w * L:(w + 1) * L] for k, w in call])
        # window w > 0 is conditioned on the last Lp INPUT frames of window w - 1, window 0 on the learnt start rows
        prev_audio = torch.stack([feats[k][w * L - Lp:w * L] if w > 0 else start_audio for k, w in call])
        indicator = (frames < p[:, 2:3]).float() if args.use_indicator else None
        out, _, _ = model.sample(audio_in, shape[idx], None if style is None else style[idx], prev_motion[idx], prev_audio,
                                 xT[idx], indicator=indicator, cfg_mode=cfg_mode, cfg_cond=cfg_cond, cfg_scale=cfg_scale,
                                 dynamic_threshold=dynamic_threshold, noise_keys=p[:, 3:5].contiguous(), timesteps=timesteps,
                                 eta=eta, solver=solver)
        prev_motion[idx] = out[:, -Lp:]
        codes[idx[:, None], rows] = out
    lengths = torch.tensor([int(n) for n in clip_lens], dtype=torch.int64)
    T_max = int(lengths.max())
    codes = codes[:, :T_max]
    keep = torch.arange(T_max, device=dev)[None, :] < lengths.to(dev)[:, None]
    return torch.where(keep[..., None], codes, torch.zeros((), device=dev)), lengths


# audio encoder batch of infer_coeffs_many: 64 clips x 10 s, the encoder batch of the configs[2] benchmark
AUDIO_BATCH_SAMPLES = 64 * 160000


@torch.no_grad()
def extract_clip_features(model, args, audios, audio_unit=640.0):
    """Audio features of many 1-D 16 kHz clips, each planned and zero-padded exactly as infer_coeffs does (plan_clip).
    The encoder runs once per group of clips with the same padded length, in batches of one clip count for every group,
    chosen so that clips x the longest padded clip stays within AUDIO_BATCH_SAMPLES: the encoder's workspace grows to
    (largest batch seen) x (longest clip seen), so a per-group count (many short clips, few long ones) would size it
    for the product of both maxima.  Returns (features: list of [n_sub_k * n_motions, d], clip_lens: list of frames to keep)."""
    plans = [plan_clip(len(a), args, audio_unit) for a in audios]
    groups = {}
    for k, (n_sub, padded, _) in enumerate(plans):
        groups.setdefault((n_sub, padded), []).append(k)
    feats = [None] * len(audios)
    step = max(1, AUDIO_BATCH_SAMPLES // max((p[1] for p in plans), default=1))
    for (n_sub, padded), ks in groups.items():
        for a in range(0, len(ks), step):
            chunk = ks[a:a + step]
            wav = torch.stack([F.pad(audios[k], (0, padded - len(audios[k])), value=0) for k in chunk])
            f = model.extract_audio_feature(wav, args.n_motions * n_sub)
            for j, k in enumerate(chunk):
                feats[k] = f[j]
    return feats, [p[2] for p in plans]


@torch.no_grad()
def infer_coeffs_many(model, args, audios, shape_coefs, style_feats, audio_unit=640.0, **queue_kwargs):
    """``infer_coeffs`` for many 1-D 16 kHz clips of any lengths: features from extract_clip_features, then
    infer_coeffs_queue.  queue_kwargs: x_T ([K, n_motions, 67] or a list; default drawn from torch's generator),
    max_clips, clip_ids, noise_seed, cfg_mode, cfg_cond, cfg_scale, dynamic_threshold (default (0, 1, 4), infer_coeffs's
    default; None turns dynamic thresholding off), timesteps, eta, solver (a respaced schedule for every clip).
    Returns (codes [K, max clip_len, 67], zero beyond each clip's length; lengths [K])."""
    K = len(audios)
    if K == 0:
        raise ValueError('infer_coeffs_many: no clips')
    feats, clip_lens = extract_clip_features(model, args, audios, audio_unit)
    queue_kwargs.setdefault('dynamic_threshold', (0, 1, 4))
    x_T = queue_kwargs.pop('x_T', None)
    if x_T is None:       # drawn on the CPU like MSMD.sample's default x_T (model.py:337)
        x_T = torch.randn((K, args.n_motions, 67)).to(model.device)
    return infer_coeffs_queue(model, args, feats, shape_coefs, style_feats, clip_lens, x_T, **queue_kwargs)


def load_model(model_root: str, model_name: str, iter_num: str, device='cuda'):
    """inference.py:85-103: <model_root>/DPT/<model_name>/{args.json, checkpoints/iter_<iter_num>.pt} ->
    (model, style_encoder, args).  The checkpoint's 'model' / 'style_enc' state_dicts load unchanged
    (same keys and shapes as the reference modules)."""
    import os
    from pathlib import Path
    from .model import get_diffusion_model
    from .style_encoder import get_style_encoder
    from .utils.model_common import load_args
    exp = Path(os.path.join(model_root, "DPT", model_name))
    model_args = load_args(exp)
    model = get_diffusion_model(model_args, device)
    ckpt = torch.load(exp / "checkpoints" / f"iter_{iter_num}.pt", map_location=device)
    style_enc = get_style_encoder(model_args, model_args.style_enc_model_style)
    style_enc.load_state_dict(ckpt['style_enc'])
    style_enc.to(device).eval()
    model.load_state_dict(ckpt['model'])
    model.eval()
    return model, style_enc, model_args


# ---------------------------------------------------------------------------------------------------------------
# Clip front-end (SURVEY section 8(f) rank 4): the numpy stages of inference.py between file I/O and the encoders,
# on the GPU through the C ABI (csrc/frontend.cu).  File decoding itself (librosa.load / pickle) stays with the caller.
def normalize_audio(audio):
    """inference.py:234: ``(audio - audio.mean()) / (audio.std() + 1e-5)`` per clip (numpy's population std).
    audio: CUDA fp32 [n] or [N, n]."""
    from . import _lib
    if audio.device.type != 'cuda':
        raise _lib.MsmdError('msmd_b200.inference.normalize_audio needs a CUDA tensor (no CPU path)')
    x = audio.detach().to(torch.float32).contiguous()
    x2 = x.reshape(1, -1) if x.ndim == 1 else x
    out = torch.empty_like(x2)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().msmd_audio_normalize(_lib.dev_ptr(x2), _lib.dev_ptr(out), x2.shape[0], x2.shape[1],
                                                   _lib.stream_ptr()))
    return out.reshape(x.shape)


def resample_linear(x, rows_out):
    """scipy ``interp1d(np.linspace(0, 1, rows_in), x, axis=0)(np.linspace(0, 1, rows_out))`` (inference.py:158-171).
    x: CUDA fp32 [rows_in, cols]."""
    from . import _lib
    if x.device.type != 'cuda':
        raise _lib.MsmdError('msmd_b200.inference.resample_linear needs a CUDA tensor (no CPU path)')
    x = x.detach().to(torch.float32).contiguous()
    if x.ndim != 2 or x.shape[0] < 1:
        raise ValueError(f'resample_linear expects [rows >= 1, cols], got {tuple(x.shape)}')
    out = torch.empty((int(rows_out), x.shape[1]), device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().msmd_resample_linear(_lib.dev_ptr(x), _lib.dev_ptr(out), x.shape[0], int(rows_out), x.shape[1],
                                                   _lib.stream_ptr()))
    return out


def prepare_style_clip(expression_coef, head_rot, coef_stats, device='cuda', original_fps=30, target_fps=25):
    """The arithmetic of ``query_for_motion_coeff`` (inference.py:108-184) on already-loaded arrays: normalise the
    expression codes and head rotations with the dataset statistics (eps 1e-9), resample original_fps -> target_fps
    by linear interpolation, concatenate.  Returns (motion_coeff [1, frames, n_exp + n_rot], shape_coef zeros [1, 100])."""
    t = lambda a: torch.as_tensor(a, dtype=torch.float32, device=device)
    exp = (t(expression_coef) - t(coef_stats['exp_mean'])) / (t(coef_stats['exp_std']) + 1e-9)
    rot = (t(head_rot) - t(coef_stats['pose_mean'])) / (t(coef_stats['pose_std']) + 1e-9)
    if original_fps is not None and original_fps != target_fps:
        new_frames = int(round(exp.shape[0] / original_fps * target_fps))
        exp, rot = resample_linear(exp, new_frames), resample_linear(rot, new_frames)
    return torch.cat([exp, rot], dim=1).unsqueeze(0), torch.zeros((1, 100), device=device)
