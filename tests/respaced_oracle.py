"""Float64 reference for sampling on respaced (DDIM) schedules, used by tests/test_respaced.py.

It is ``oracle.denoiser.sample`` with the update coefficients of a respaced schedule: the network forward and the CFG
entries come from the oracle unchanged, only the loop over timesteps and the update differ."""
import torch

from oracle.denoiser import cfg_entries, denoiser_forward


def sample_respaced(sd, cfg, audio_feat, shape_coef_or_feat, style_feat, timesteps, eta, prev_motion=None,
                    prev_audio=None, x_T=None, z=None, indicator=None, cfg_mode=None, cfg_cond=None, cfg_scale=1.15,
                    ret_traj=False, n_steps=None, t_start=None, dynamic_threshold=None, separate=False):
    """``sample`` on a respaced (DDIM) schedule: visits the strictly decreasing ``timesteps`` (from ``t_start``, default
    the first entry, for ``n_steps`` entries) with eta in [0, 1].  Per visited t with successor s (0 after the last entry),
    A = alpha_bars[t], B = alpha_bars[s] (alpha_bars[0] = 1), all in float64 from the schedule buffers:
      sigma = eta sqrt((1 - B)/(1 - A)) sqrt(1 - A/B),  r = sqrt(max(0, 1 - B - sigma^2))
      'sample': k = r / sqrt(1 - A);  x_s = k x_t + (sqrt(B) - sqrt(A) k) x0_hat + sigma z_t
      'noise':  x_s = sqrt(B/A) x_t + (r - sqrt(B) sqrt(1 - A)/sqrt(A)) eps_hat + sigma z_t
    z_t = z[t] (or torch.randn) is drawn only when s > 0.  The network output is the CFG-combined, optionally thresholded
    output of ``sample``.  With separate=True the cumulative static part sums the output coefficient times the static
    part.  Returns like ``sample``; ret_traj gives {t: x_t} over the visited t and the last successor; the state stays
    float64."""
    N = audio_feat.shape[0]
    sched = {k[len('diffusion_sched.'):]: v for k, v in sd.items() if k.startswith('diffusion_sched.')}
    ab = sched['alpha_bars'].double()
    ts = [int(t) for t in timesteps]
    cfg_mode = cfg_mode or cfg.cfg_mode
    if cfg_cond is None:
        cfg_cond = [c for c in cfg.guiding_conditions.split(',') if c in ('style', 'audio')]
    cfg_cond = [c for c in cfg_cond if c in ('audio', 'style')]
    if not isinstance(cfg_scale, list):
        cfg_scale = [cfg_scale] * len(cfg_cond)
    if cfg_cond:
        cfg_cond, cfg_scale = zip(*sorted(zip(cfg_cond, cfg_scale), key=lambda x: ['audio', 'style'].index(x[0])))
    shape_feat = shape_coef_or_feat
    if style_feat is None:
        style_feat = sd['null_style_feat'].expand(N, -1, -1)
    if shape_feat.ndim == 2:
        shape_feat = shape_feat.unsqueeze(1)
    if style_feat.ndim == 2:
        style_feat = style_feat.unsqueeze(1)
    if prev_motion is None:
        prev_motion = sd['start_motion_feat'].expand(N, -1, -1)
    if prev_audio is None:
        prev_audio = sd['start_audio_feat'].expand(N, -1, -1)
    if x_T is None:
        x_T = torch.randn(N, cfg.n_motions, 67)
    audio_in, person_in = cfg_entries(sd, cfg, audio_feat, shape_feat, style_feat, cfg_mode, cfg_cond)
    E = len(audio_in)
    audio_in = torch.cat(audio_in, 0)
    person_in = torch.cat(person_in, 0)
    pm = torch.cat([prev_motion] * E, 0)
    pa = torch.cat([prev_audio] * E, 0)
    ind = torch.cat([indicator] * E, 0) if indicator is not None else None
    st = torch.cat([style_feat] * E, 0)
    fn = lambda *a: denoiser_forward(sd, cfg, *a, keep_separate=separate)
    pos = ts.index(t_start if t_start is not None else ts[0])
    visit = ts[pos:pos + n_steps] if n_steps else ts[pos:]
    x = x_T.double()
    cum_static = torch.zeros_like(x)
    alpha_traj, tgt_dyn = [], None
    traj = {visit[0]: x_T}
    for t in visit:
        i = ts.index(t)
        s = ts[i + 1] if i + 1 < len(ts) else 0
        A, B = ab[t], (ab[s] if s > 0 else torch.ones((), dtype=torch.float64))
        sigma = eta * torch.sqrt((1 - B) / (1 - A)) * torch.sqrt(torch.clamp(1 - A / B, min=0))
        r = torch.sqrt(torch.clamp(1 - B - sigma ** 2, min=0))
        zt = (z[t] if z is not None else torch.randn_like(x_T)).double() if s > 0 else torch.zeros_like(x)
        step = torch.full((N * E,), t, dtype=torch.long)
        res = fn(torch.cat([x.float()] * E, 0), audio_in, person_in, st, pm, pa, step, ind)
        if separate:
            dyn, stat_b, alph = res
            face = torch.einsum('nlb,nbc->nlc', alph, stat_b[:, :, :-3])
            pose = stat_b[:, :, -3:].sum(1, keepdim=True).expand(-1, dyn.shape[1], -1)
            stat = torch.cat([face, pose], -1)
            res = dyn + stat
        if dynamic_threshold:
            q, lo, hi = dynamic_threshold
            a = res[:, -cfg.n_motions:].reshape(N * E, -1).abs()
            thr = torch.clamp(torch.quantile(a, q, dim=1), min=lo, max=hi)[:, None, None]
            res = torch.clamp(res, min=-thr, max=thr)

        def combine(parts):   # the CFG recursion of sample, aliasing included
            parts = [c[:, -cfg.n_motions:] for c in parts]
            acc = parts[0]
            for k in range(E - 1):
                ref_k = acc if (cfg_mode == 'independent' or k == 0) else parts[k]
                acc = acc + cfg_scale[k] * (parts[k + 1] - ref_k)
            return acc
        tgt = combine(res.chunk(E)).double()
        if cfg.target == 'noise':
            c0 = torch.sqrt(B / A)
            c1 = r - torch.sqrt(B) * torch.sqrt(1 - A) / torch.sqrt(A)
        else:
            c0 = r / torch.sqrt(1 - A)
            c1 = torch.sqrt(B) - torch.sqrt(A) * c0
        x = c0 * x + c1 * tgt + sigma * zt
        if separate:
            tgt_dyn = combine(dyn.chunk(E))
            cum_static = cum_static + c1 * combine(stat.chunk(E)).double()
            alpha_traj.append(combine(alph.chunk(E)))
        traj[s] = x
    if ret_traj:
        return traj, x_T, audio_feat
    if separate:
        return x, x_T, audio_feat, tgt_dyn, cum_static, torch.cat(alpha_traj, 0)
    return x, x_T, audio_feat
